#!/usr/bin/env python
"""bench.py — BASELINE.json metric: "edges/sec in F-gradient step at 1/2/4/8 B200; iters/sec on
com-amazon K=200".

A step = one call of the hot path (backtrackingLineSearchs, codes/bigclam4-7.scala:152-223: PRE +
16-candidate line search + row swap + sumF update + LLH) over the whole graph.  Default workload
(`--config amazon200`, BASELINE config 3): the com-amazon topology (SNAP, 334,863 nodes / 925,872
edges, package data bigclam_apachespark_b200/data/graphs/com-amazon.npz) with K=200 and the synthetic
F0 of BASELINE.md (U[0,1) with probability 0.05, seed 1234), fp64.  The other BASELINE configs are
`--config enron50 | amazon500 | rmat` (or --graph / --k).

F lives on the device as SPARSE ROWS (the reference's own layout, RDD[(Long, BSV[Double])],
bigclam4-7.scala:97-104); `--layout dense` selects the round-1 dense n x K kernels.  The roofline
is reported against SURVEY §8(d)'s DENSE-model algorithmic bytes (nnz*(K*8+4) + N*(2*K*8+8) + K*8);
`layout_bytes_per_launch` is what the sparse layout really has to move and `traffic` the DRAM bytes
of one launch measured in this run by a side process under ncu (never inside the timed region).
The working set of the sparse layout is ~80 MB: it is L2-resident on purpose, nothing is flushed.

  value   directed neighbour-list entries processed per second (= 2 x undirected edges), F resident
          in HBM, K steps run by the device-side loop (bigclam_run), CUDA events on the launching stream
  e2e     the same metric through per-call bigclam_step() with host buffers (uset mask H2D from
          pinned memory, LLH/n_updated D2H every step)
  roofline  algorithmic bytes of one step kernel / its average duration (CUDA events in the library)
  cpu_baseline  the CPU restatement of the reference (oracle/, NOT Spark) on the host cores
  line_search   the default engine evaluates a candidate step only if a bound on the node's objective cannot exclude it
          (same accepted steps, rows and LLH as the reference's exhaustive 16 candidates: tests/test_gpu_prune.py); this
          block says how many nodes were line-searched in the timed steps and times, beside the headline and never as
          the headline, the exhaustive engine (BIGCLAM_F_LS_EXHAUSTIVE) on the same steps and a whole SGDFindC run from
          the synthetic F0 to the reference's stop rule
`--impl reference` times that CPU restatement alone (the reference needs a JVM + Spark: absent).
`--dump-outputs DIR` writes what the timed steps computed (dump_outputs), so that two builds can be compared on the same
inputs: the graph and F0 are seeded, identical from run to run for the same arguments.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True            # the benchmark leaves the tree it runs from as it found it

CONFIGS = {
    "enron50": dict(graph="email-enron", k=50, note="BASELINE config 2 (Email-Enron, reciprocal lines deduplicated)"),
    "amazon200": dict(graph="com-amazon", k=200, note="BASELINE config 3 (headline)"),
    "amazon500": dict(graph="com-amazon", k=500, note="BASELINE config 4"),
    "rmat": dict(graph="rmat:10000000:100000000", k=1000, note="BASELINE config 5 (R-MAT 10M nodes / 100M edges)"),
}


def workload_name(graph, k):
    return f"{graph} K={k}, synthetic F0 (p=0.05 U[0,1), seed 1234), fp64"


def load_graph(graph):
    from bigclam_apachespark_b200 import graphs as G
    if graph.startswith("rmat:"):
        _, nn, mm = graph.split(":")
        if int(mm) >= 20_000_000:            # big synthetic graphs: generated on the GPU when there is one (plumbing)
            try:
                import torch
                if torch.cuda.is_available():
                    return G.rmat_graph_torch(int(nn), int(mm), seed=42, device=f"cuda:{torch.cuda.current_device()}")
            except ImportError:
                pass
            return G.rmat_graph_fast(int(nn), int(mm), seed=42)
        return G.rmat_graph(int(nn), int(mm), seed=42)
    rp, col, _ = G.load_npz_graph(graph)
    return rp, col


def load_workload(graph, k):
    """(rowptr, col, F0): F0 dense when n x K fits comfortably, else a scipy CSR matrix (same distribution)."""
    from bigclam_apachespark_b200 import graphs as G
    rp, col = load_graph(graph)
    n = len(rp) - 1
    if n * k > (1 << 29):
        import scipy.sparse as sps
        gen = G.synthetic_F0_csr_stratified if n * k > (1 << 32) else G.synthetic_F0_csr
        if n * k > (1 << 32):
            try:
                import torch
                if torch.cuda.is_available():
                    gen = lambda n_, k_, seed, density: G.synthetic_F0_csr_stratified_torch(      # noqa: E731
                        n_, k_, seed=seed, density=density, device=f"cuda:{torch.cuda.current_device()}")
            except ImportError:
                pass
        ip, ix, vl = gen(n, k, seed=1234, density=0.05)
        return rp, col, sps.csr_matrix((vl, ix, ip), shape=(n, k))
    return rp, col, G.synthetic_F0(n, k, seed=1234, density=0.05)


def base_config(graph, k, n, nnz, layout):
    """The same keys in both arms (GPU and reference)."""
    return {"workload": workload_name(graph, k), "graph": graph, "k": int(k), "n": int(n), "nnz_directed": int(nnz),
            "edges_undirected": int(nnz // 2), "f0": "synthetic p=0.05 U[0,1) seed 1234", "f_layout": layout}


def alg_bytes(n, nnz, k, s=8):
    """SURVEY.md §8(d): nnz*(K*s+4) + N*(2*K*s+8) + K*s."""
    return nnz * (k * s + 4) + n * (2 * k * s + 8) + k * s


def hbm_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region through NVML (the same counters
    `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints), every ~5 ms from a thread."""

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def start(self):
        try:
            import pynvml as N
            N.nvmlInit()
            self.N = N
            self.h = N.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(self.h, N.NVML_CLOCK_SM))
        except Exception as exc:            # noqa: BLE001
            self.N = None
            self.err = repr(exc)
            return
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def _run(self):
        N = self.N
        bits = {"hw_slowdown": N.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": N.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": N.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": N.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.samples.append(float(N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM)))
                r = N.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:               # noqa: BLE001
                pass
            time.sleep(0.005)

    def stop(self):
        if self.N is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self._stop.set()
        self._t.join(timeout=1)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU restatement of the reference (oracle/): the cpu_baseline leg and the --impl reference arm
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_oracle_all_cores():
    """torchrun exports OMP_NUM_THREADS=1 to its children: the oracle must see the box's cores anyway (libgomp reads
    the variable when the library is loaded)."""
    os.environ["OMP_NUM_THREADS"] = str(host_cores())
    os.environ.pop("OMP_THREAD_LIMIT", None)
    from oracle import oracle as O
    O.build()
    return O


def time_oracle(rp, col, F0, k, steps, warmup, budget_s=200.0):
    """Faithful CPU restatement (all 16 candidates per node, like the reference); all host threads.  A step is the
    whole graph when the run fits the time budget; otherwise a fixed sample of the nodes (uset) per step, with the
    metric counted over the sample's neighbour-list entries.  Returns (edges per second, cores, sample text)."""
    O = load_oracle_all_cores()
    P = O.make_params(k)
    if hasattr(F0, "toarray"):
        raise RuntimeError("the CPU restatement needs a dense F0")
    n = len(rp) - 1
    deg = np.diff(rp)
    F, s = F0, O.colsum(F0)
    t0 = time.perf_counter()
    r = O.step(rp, col, F, s, P, early_exit=False)           # probe: one full step (also the first warm-up step)
    probe = time.perf_counter() - t0
    F, s = r.F, r.sumF
    total_steps = steps + max(warmup, 1)
    mask, frac, sample = None, 1.0, f"{steps} full steps of the workload (all 16 candidates per node), {max(warmup, 1)} warm-up"
    if probe * total_steps > budget_s:
        frac = max(budget_s / (probe * total_steps), 1.0 / 64.0)
        rng = np.random.default_rng(99)
        mask = (rng.random(n) < frac).astype(np.uint8)
        sample = (f"{steps} steps over a fixed {100 * mask.mean():.1f} % node sample (uset, {int(deg[mask != 0].sum())} neighbour-list entries; "
                  f"all 16 candidates per node; the LLH pass after each step still covers the whole graph), {max(warmup, 1)} warm-up; "
                  f"one full step took {probe:.2f} s")
    edges = int(deg.sum()) if mask is None else int(deg[mask != 0].sum())
    times = []
    for i in range(total_steps - 1):
        t0 = time.perf_counter()
        r = O.step(rp, col, F, s, P, node_mask=mask, early_exit=False)
        dt = time.perf_counter() - t0
        if i >= max(warmup, 1) - 1:
            times.append(dt)
        F, s = r.F, r.sumF
    sec = float(np.mean(times)) if times else probe
    return edges / sec, O.num_threads(), sample, sec


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rp, col, F0 = load_workload(args.graph, args.k)
    n, nnz = len(rp) - 1, len(col)
    val, cores, sample, sec = time_oracle(rp, col, F0, args.k, args.steps, args.warmup)
    print(json.dumps({
        "impl": "reference", "metric": "edges/sec in F-gradient step", "value": val, "unit": "edges/s",
        "unit_note": "directed neighbour-list entries per second (2 per undirected edge)",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "iters_per_sec": 1.0 / sec, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "SNAP topology (package data) or generated R-MAT + synthetic F0",
        "config": base_config(args.graph, args.k, n, nnz, args.layout),
        "note": "CPU restatement of the reference (oracle/, C + OpenMP, -O3 -march=native), NOT Spark: no JVM in the image. PARITY UNPINNED.",
        "cpu_baseline": {"value": val, "unit": "edges/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------
def measure_traffic(args, kernel_regex):
    """DRAM bytes of ONE launch of the step kernel, measured now by a side process under ncu (same workload, same
    library); None when ncu is not available.  Never overlaps the timed region."""
    if args.no_traffic:
        return None, "skipped (--no-traffic)"
    cmd = ["ncu", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k", f"regex:{kernel_regex}",
           "--launch-skip", "4", "--launch-count", "1", "--csv", sys.executable, os.path.join(REPO, "tools", "profile_step.py"),
           str(args.k), "5", "2", args.graph]
    env = dict(os.environ, BIGCLAM_AB_SPARSE="1" if args.layout == "sparse" else "0", PYTHONDONTWRITEBYTECODE="1")
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=180, env=env).stdout
    except Exception as exc:                # noqa: BLE001
        return None, f"ncu failed: {exc!r}"
    tot = 0.0
    seen = 0
    for line in out.splitlines():
        if "dram__bytes_" in line:
            parts = [p.strip('"') for p in line.split('","')]
            try:
                v = float(parts[-1].replace(",", ""))
                unit = parts[-2].lower()
            except ValueError:
                continue
            mult = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, None)
            if mult is None:
                continue
            tot += v * mult
            seen += 1
    if seen < 2:
        return None, "ncu gave no dram__bytes rows"
    return int(tot), "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu side process in this run"


def sparse_layout_bytes(indptr, rp, col):
    """Bytes the sparse layout has to move per launch: every neighbour's row block once per edge (+ its 8-byte header
    and the 4-byte neighbour id), every own row block read once and written once (+ header each way)."""
    cnt = np.diff(indptr)
    blk = 8 * ((cnt + 1) // 2 * 2) + 2 * ((cnt + 7) // 8 * 8)
    return int(blk[col].sum() + 12 * len(col) + 2 * blk.sum() + 16 * (len(rp) - 1))


DUMP_F_BYTES = 32 << 20                      # F.npy; with llh.npy and sumF.npy the dump stays below 64 MB


def dump_outputs(out_dir, b, llh):
    """Writes what the hot path hands its caller after the last timed step, as float64 .npy files: llh (the LLH of that
    step), sumF (K) and F.  F is n x K; when that exceeds DUMP_F_BYTES, the rows of a fixed sample (seed 0, ascending
    node ids) stand for it, the same rows in every run of the same workload.  Returns a description for the JSON line."""
    import scipy.sparse as sps
    indptr, indices, values = b.F_csr()
    n, k = len(indptr) - 1, b.K
    m = min(n, DUMP_F_BYTES // (8 * k))
    rows = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    F = sps.csr_matrix((values, indices, indptr), shape=(n, k))[rows].toarray()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "llh.npy"), np.array([llh], dtype=np.float64))
    np.save(os.path.join(out_dir, "sumF.npy"), b.sumF)
    np.save(os.path.join(out_dir, "F.npy"), F)
    return {"dir": out_dir, "files": ["llh.npy", "sumF.npy", "F.npy"],
            "F_rows": "all" if m == n else f"{m} of {n} rows, np.random.default_rng(0).choice(n, {m}, replace=False), sorted"}


class ExtrasWatchdog:
    """The headline numbers (value, roofline, e2e) are measured first; everything after them (the reference-style-init
    workload, the exhaustive-line-search arm, the run to convergence, the ncu side process, the CPU baseline) explains them.
    If that part stalls — a wedged side process, a stuck device call — the line measured so far is printed with
    `extras_cut` set and the process ends, instead of the whole run being lost at the caller's limit."""

    def __init__(self, limit_s):
        self.limit_s = limit_s
        self.lock = threading.Lock()
        self.line = None
        self.stage = "start"
        self.printed = False
        self.timer = None

    def arm(self, line):
        self.line = line
        self.timer = threading.Timer(self.limit_s, self._fire)
        self.timer.daemon = True
        self.timer.start()

    def _fire(self):
        with self.lock:
            if self.printed:
                return
            self.printed = True
            out = dict(self.line, extras_cut=f"stopped after {self.limit_s:.0f} s in '{self.stage}': fields not reached are null")
            sys.stdout.write(json.dumps(out) + "\n")
            sys.stdout.flush()
        os._exit(0)

    def emit(self, line):
        with self.lock:
            if self.printed:
                return
            self.printed = True
            if self.timer is not None:
                self.timer.cancel()
            print(json.dumps(line), flush=True)


def run_single(args):
    import torch
    from bigclam_apachespark_b200 import BigClam, _lib

    torch.cuda.set_device(0)
    K = args.k
    rp, col, F0 = load_workload(args.graph, K)
    n, nnz = len(rp) - 1, len(col)
    sparse = args.layout == "sparse"
    b = BigClam(device=0, time_kernels=True, sparse_rows=sparse)
    b.set_graph(rp, col).set_K(K)
    stream = torch.cuda.current_stream()
    b.set_stream(stream.cuda_stream)
    b.set_F(F0)

    # ---- value: device-resident loop ----
    b._run(4, 0.0, args.warmup)                      # W untimed warm-up steps
    if sparse:
        for _ in range(3):                           # (still untimed) let the tile cut settle on this workload's rows
            b.retile()
            b._run(4, 0.0, 2)
        b.tile_stats()                               # reset the counters
        b.ls_stats()
    sampler = ClockSampler(0)
    sampler.start()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    b._run(4, 0.0, args.steps)                       # exactly K steps (rel_tol 0: never converges early)
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    assert b.last_calls == args.steps
    total_ms = e0.elapsed_time(e1)
    kern_ms, n_step_kernels, n_all = b.kernel_time()
    ms_per_step = total_ms / args.steps
    value = nnz / (ms_per_step * 1e-3)
    llh_end = float(b.last_trace[-1])
    tiles = b.tile_stats() if sparse else None
    ls = b.ls_stats() if sparse else None
    dumped = dump_outputs(args.dump_outputs, b, llh_end) if args.dump_outputs else None    # before e2e moves F on

    # ---- roofline of the dominant kernel ----
    peak, peak_src = hbm_peak()
    balg = alg_bytes(n, nnz, K)
    kavg_ms = kern_ms / max(n_step_kernels, 1)
    achieved = balg / (kavg_ms * 1e-3) / 1e9
    kernel = "tile_step_kernel" if sparse else "step_kernel"
    layout_bytes = sparse_layout_bytes(b.F_csr()[0], rp, col) if sparse else balg

    # ---- e2e: per-call C ABI with host buffers ----
    mask = torch.ones(n, dtype=torch.uint8).pin_memory()
    llh = C.c_double(); nupd = C.c_int64()
    lib = _lib.load()
    for _ in range(3):
        _lib.check(lib.bigclam_step(b._ctx, mask.data_ptr(), C.byref(llh), C.byref(nupd)), b._ctx)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _lib.check(lib.bigclam_step(b._ctx, mask.data_ptr(), C.byref(llh), C.byref(nupd)), b._ctx)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    e2e = {"value": nnz / (e2e_ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": int(n),
           "d2h_bytes_per_step": 72, "ms_per_step": e2e_ms,
           "note": "bigclam_step() per step: uset mask H2D (pinned) + sumF commit + the next call's step kernel launched speculatively (its PRE is this call's LLH) + LLH/n_updated D2H, synchronous; F stays resident like the reference's cached RDD"}

    # ---- the line as measured so far; what follows explains it and cannot lose it (ExtrasWatchdog) ----
    cfg = base_config(args.graph, K, n, nnz, args.layout)
    line = {
        "metric": "edges/sec in F-gradient step", "value": value, "unit": "edges/s",
        "unit_note": "directed neighbour-list entries per second (2 per undirected edge)", "value_undirected_edges_per_s": value / 2,
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "untimed_steps_before_timing": args.warmup + (6 if sparse else 0),
        "iters_per_sec": 1e3 / ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "SNAP topology (package data) or generated R-MAT + synthetic F0",
        "config": cfg, "parallelism": "1 GPU",
        "l2": ("sparse rows: working set ~2 x %.0f MB, L2-resident by design, no flush" % (layout_bytes / 4e6)) if sparse
              else "inputs (F, 2 buffers) larger than L2, no flush",
        "llh_end": llh_end, "parity": "PARITY UNPINNED: checked against oracle/ (CPU restatement), not against outputs of the reference",
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(n_all), "dumped_outputs": dumped,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "traffic_source": "not reached", "kernel": kernel,
                     "kernel_ms": kavg_ms, "alg_bytes_per_launch": balg, "peak_source": peak_src,
                     "f_layout": args.layout, "layout_bytes_per_launch": layout_bytes,
                     "layout_frac": layout_bytes / (kavg_ms * 1e-3) / 1e9 / peak,
                     "note": "achieved/frac use SURVEY 8(d)'s dense-model algorithmic bytes; layout_bytes_per_launch is what the sparse rows move, traffic what DRAM saw (the rest is L2)",
                     "tiles": tiles},
        "cpu_baseline": None, "reference_init_workload": None, "line_search": None,
    }
    dog = ExtrasWatchdog(args.extras_limit)
    dog.arm(line)

    # ---- DRAM traffic of one launch, measured now (side process under ncu) ----
    dog.stage = "roofline.traffic (ncu side process)"
    traffic, traffic_src = measure_traffic(args, kernel)
    line["roofline"]["traffic"] = traffic
    line["roofline"]["traffic_source"] = traffic_src

    # ---- CPU baseline beside it (bounded: 5 faithful steps after 1 warm-up) ----
    dog.stage = "cpu_baseline"
    if not args.no_cpu and not hasattr(F0, "tocsr"):
        try:
            val, cores, sample, sec = time_oracle(rp, col, F0, K, 5, 1, budget_s=45.0)
            line["cpu_baseline"] = {"value": val, "unit": "edges/s", "cores": cores, "kind": "port",
                                    "sample": sample + "; CPU restatement of the reference (oracle/, -O3 -march=native), not Spark",
                                    "ms_per_step": sec * 1e3}
        except Exception as exc:            # noqa: BLE001
            line["cpu_baseline"] = {"unavailable": repr(exc)}

    # ---- workload A of SURVEY §8d: the reference's own init (conductance seeds, 0/1 indicator columns) ----
    dog.stage = "reference_init_workload"
    try:
        if not args.no_init_a and not hasattr(F0, "tocsr") and n <= 2_000_000:
            t0 = time.perf_counter()
            b.initNeighborComF(K)
            init_s = time.perf_counter() - t0
            b._run(4, 0.0, args.warmup)
            torch.cuda.synchronize()
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record(stream)
            b._run(4, 0.0, args.steps)
            eb.record(stream)
            torch.cuda.synchronize()
            ms_a = ea.elapsed_time(eb) / args.steps
            kms_a, nk_a, _ = b.kernel_time()
            line["reference_init_workload"] = {
                "workload": f"{args.graph} K={K}, F0 = initNeighborComF({K}) (bigclam4-7.scala:81-108: 0/1 indicator columns of the best-conductance seeds)",
                "value": nnz / (ms_a * 1e-3), "unit": "edges/s", "ms_per_step": ms_a, "step_kernel_ms": kms_a / max(nk_a, 1),
                "roofline_frac": balg / (kms_a / max(nk_a, 1) * 1e-3) / 1e9 / peak, "init_seconds": init_s,
                "llh_end": float(b.last_trace[-1])}
    except Exception as exc:                # noqa: BLE001
        line["reference_init_workload"] = {"unavailable": repr(exc)}
    try:
        b.close()
    except Exception:                       # noqa: BLE001
        pass

    # ---- the same steps with the exhaustive line search (all 16 candidates of every node, like the reference's cartesian,
    #      bigclam4-7.scala:172-181; BIGCLAM_F_LS_EXHAUSTIVE).  The default engine skips candidates that a bound proves unable
    #      to pass the Armijo test — same accepted steps, same rows, same LLH bits (tests/test_gpu_prune.py); this is the
    #      price of evaluating them anyway, measured beside it (not the headline).
    if sparse and not args.no_line_search:
        line_search = {"mode": "bounds (default): a candidate step is evaluated only if a bound on the node's objective cannot exclude it",
                       "nodes_asked": ls["nodes_asked"], "nodes_line_searched": ls["nodes_searched"],
                       "exhaustive": None, "run_to_convergence": None}
        line["line_search"] = line_search
        dog.stage = "line_search.exhaustive"
        try:
            bx = BigClam(device=0, time_kernels=True, sparse_rows=True, exhaustive_linesearch=True)
            bx.set_graph(rp, col).set_K(K)
            bx.set_stream(stream.cuda_stream)
            bx.set_F(F0)
            bx._run(4, 0.0, args.warmup)
            for _ in range(3):
                bx.retile()
                bx._run(4, 0.0, 2)
            torch.cuda.synchronize()
            x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            x0.record(stream)
            bx._run(4, 0.0, args.steps)
            x1.record(stream)
            torch.cuda.synchronize()
            xk_ms, xk_n, _ = bx.kernel_time()
            x_llh = float(bx.last_trace[-1])
            bx.close()
            x_ms = x0.elapsed_time(x1) / args.steps
            line_search["exhaustive"] = {"ms_per_step": x_ms, "step_kernel_ms": xk_ms / max(xk_n, 1),
                                         "value": nnz / (x_ms * 1e-3), "llh_end": x_llh,
                                         "llh_rel_diff_vs_default": abs(x_llh - llh_end) / abs(llh_end),
                                         "roofline_frac": balg / (xk_ms / max(xk_n, 1) * 1e-3) / 1e9 / peak}
        except Exception as exc:            # noqa: BLE001
            line_search["exhaustive"] = {"unavailable": repr(exc)}
        # the whole solver run from this F0 as the reference would do it (SGDFindC, :225-243: until |1 - new/old| < 1e-4):
        # the early iterations, where most nodes still move and the bounds exclude the least, are in here
        dog.stage = "line_search.run_to_convergence"
        try:
            bc = BigClam(device=0, time_kernels=True, sparse_rows=True)
            bc.set_graph(rp, col).set_K(K)
            bc.set_stream(stream.cuda_stream)
            bc.set_F(F0)
            bc.ls_stats()
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            bc.SGDFindC(rel_tol=1e-4, max_outer=500)
            c1.record(stream)
            torch.cuda.synchronize()
            conv_calls = int(bc.last_calls)
            conv_ls = bc.ls_stats()
            bc.close()
            line_search["run_to_convergence"] = {
                "calls": conv_calls, "ms_total": c0.elapsed_time(c1), "ms_per_call": c0.elapsed_time(c1) / max(conv_calls, 1),
                "nodes_asked": conv_ls["nodes_asked"], "nodes_line_searched": conv_ls["nodes_searched"],
                "note": "SGDFindC from the synthetic F0 to the reference's stop rule (rel_tol 1e-4), cold start: tile cut and pool sizes settle inside"}
        except Exception as exc:            # noqa: BLE001
            line_search["run_to_convergence"] = {"unavailable": repr(exc)}

    dog.emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="amazon200", choices=sorted(CONFIGS), help="BASELINE.json config (default: the headline)")
    ap.add_argument("--k", type=int, default=None, help="number of communities (overrides --config)")
    ap.add_argument("--graph", default=None, help="fixture name or rmat:<nodes>:<edges> (overrides --config)")
    ap.add_argument("--layout", default="sparse", choices=["dense", "sparse"],
                    help="device layout of F: sparse rows like the reference's BSV[Double] (default), or dense n x K rows")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-init-a", action="store_true", help="skip the reference-style-init extra workload")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu side process that measures DRAM traffic")
    ap.add_argument("--no-line-search", action="store_true", help="skip the exhaustive-line-search arm and the run to convergence")
    ap.add_argument("--extras-limit", type=float, default=420.0,
                    help="seconds the explanatory legs after the timed regions may take before the line is printed without them")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed (llh, sumF, F or a fixed sample of its rows) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is implemented for the single-GPU arm (--impl b200 --gpus 1)")
    cfg = CONFIGS[args.config]
    args.graph = args.graph or cfg["graph"]
    args.k = args.k or cfg["k"]
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    if args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1:
        from bigclam_apachespark_b200 import dist
        return dist.bench_main(args, load_workload, alg_bytes, hbm_peak, ClockSampler, base_config)
    return run_single(args)


if __name__ == "__main__":
    main()
