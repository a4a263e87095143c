"""Kernel LOGIC of the sparse-row engine on the CPU (no GPU in this container): a selection of the `-m gpu` tests of
tests/test_gpu_sparse.py is run, in a child pytest, against the HOST-EMULATION build of the whole C API
(tests/emu/build_hostemu.sh: csrc/bigclam_capi.cu + the kernel sources compiled for the host against the SIMT
emulation of tests/emu/include/cuda_emu.h — one OS thread per CUDA thread, warp collectives as barrier rounds, so a
collective reached by part of a warp hangs instead of passing).  The tile path, the general path, split hubs, the
fixed-order reduction, the pool / CSR entry points and the device-side loop bookkeeping all run here against the
oracle.  Test infrastructure only: the product library has no CPU path and the `-m gpu` tests on the B200 remain
the parity tests of the compiled sm_100a code."""
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SELECTION = ("golden_tiny or uset_mask or csr_entry or pool_exhaustion or split_hubs or mode_limits or "
             "(all_k and (k1- or 3 or 31 or 65))")


def _child(test_file, selection, nobuild):
    env = dict(os.environ, BIGCLAM_HOSTEMU="1")
    if nobuild:
        env["BIGCLAM_HOSTEMU_NOBUILD"] = "1"
    else:
        env.pop("BIGCLAM_HOSTEMU_NOBUILD", None)
    cmd = [sys.executable, "-m", "pytest", os.path.join(REPO, "tests", test_file), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider"]
    if selection:
        cmd += ["-k", selection]
    r = subprocess.run(cmd, cwd=REPO, env=env, capture_output=True, text=True, timeout=1400)
    tail = "\n".join((r.stdout + r.stderr).splitlines()[-25:])
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail


@pytest.mark.timeout(1500)
def test_sparse_engine_under_host_emulation():
    _child("test_gpu_sparse.py", SELECTION, nobuild=False)


@pytest.mark.timeout(1500)
def test_multi_gpu_c_abi_under_host_emulation():
    """bigclam_multi_* on 2 and 3 emulated devices: node deal, pool regions, peer pushes, the fused collective (publish,
    flags, rank-ordered sums), the device-side loop on every rank — against the oracle, replicas bit-identical."""
    _child("test_gpu_multi.py", None, nobuild=True)
    _child("test_hostemu_multirank.py", None, nobuild=True)


@pytest.mark.timeout(900)
def test_line_search_bounds_under_host_emulation():
    """Line search by bounds (csrc/bigclam_tile.cuh H2, bigclam_sparse.cuh bound_mask) against the exhaustive search and the
    oracle: the same accepted steps, F, sumF and LLH bits — a selection of tests/test_gpu_prune.py (large-graph regime through
    an injected sumF, values next to the clamps)."""
    _child("test_gpu_prune.py", "(random_graphs and 900) or clamped", nobuild=True)


@pytest.mark.timeout(600)
def test_c_caller_gpu_tests_under_host_emulation():
    """The `-m gpu` tests of the plain-C caller (tests/test_gpu_zy_c_host.py), linked with the emulation build: the init mode
    against the Python driver bit for bit.  (The C caller, the JNI shim and the C++ mirror against the oracle run in the CPU suite
    themselves — tests/test_c_host.py, test_jni_shim.py, test_cpp_host.py link the emulation build directly; the other `-m gpu` tests
    of that file were run under BIGCLAM_HOSTEMU=1 by hand when they were written.)"""
    _child("test_gpu_zy_c_host.py", "init_mode", nobuild=True)


@pytest.mark.timeout(600)
def test_conductance_kernel_under_host_emulation():
    _child("test_gpu_init.py", "twin and (80 or 300) or unsorted", nobuild=True)


def _bench_dryrun(*flags):
    import json
    if not os.path.exists(os.path.join(REPO, "tests", "emu", "libbigclam_hostemu.so")):
        subprocess.run([os.path.join(REPO, "tests", "emu", "build_hostemu.sh")], check=True)
    cmd = [sys.executable, os.path.join(REPO, "tests", "emu", "bench_dryrun.py"), "--graph", "rmat:150:500", "--k", "16",
           "--steps", "2", "--warmup", "3", "--no-traffic", *flags]
    r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=800)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]                  # ONE JSON line, whatever happens after the timed regions
    return json.loads(lines[0])


@pytest.mark.timeout(900)
def test_bench_single_gpu_arm_dry_run():
    """Control flow of bench.run_single (every leg and the JSON contract) on a tiny graph: the library is the host-emulation
    build and torch.cuda's stream / event calls are host stand-ins (tests/emu/bench_dryrun.py).  No number in it means
    anything; the keys, their consistency and the one-line rule do."""
    d = _bench_dryrun()
    assert d["metric"] == "edges/sec in F-gradient step" and d["unit"] == "edges/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["untimed_steps_before_timing"] == 3 + 6          # warm-up + the steps over which the tile cut settles (both arms)
    assert set(d["config"]) == {"workload", "graph", "k", "n", "nnz_directed", "edges_undirected", "f0", "f_layout"}
    assert abs(d["value"] - d["config"]["nnz_directed"] / (d["ms_per_step"] * 1e-3)) <= 1e-9 * d["value"]
    assert d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] == d["config"]["n"] and d["e2e"]["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["kernel"] == "tile_step_kernel" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
    assert rf["alg_bytes_per_launch"] == 1000 * (16 * 8 + 4) + 150 * (2 * 16 * 8 + 8) + 16 * 8      # SURVEY 8(d)
    assert rf["layout_bytes_per_launch"] > 0 and rf["tiles"]["tiles_done"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert d["reference_init_workload"]["llh_end"] < 0
    ls = d["line_search"]
    assert 0 < ls["nodes_line_searched"] <= ls["nodes_asked"]
    assert ls["exhaustive"]["llh_rel_diff_vs_default"] <= 1e-13 and ls["run_to_convergence"]["calls"] > 0
    assert "extras_cut" not in d


@pytest.mark.timeout(900)
def test_bench_prints_its_line_when_an_explanatory_leg_stalls():
    """The headline (value, roofline, e2e) is measured first; a leg after it that exceeds --extras-limit ends the run with
    the line measured so far (exit code 0, `extras_cut` says where) instead of losing it at the caller's limit."""
    d = _bench_dryrun("--extras-limit", "2")
    assert "extras_cut" in d and d["value"] > 0 and d["e2e"]["value"] > 0 and d["roofline"]["frac"] > 0
    assert d["line_search"] is None or d["line_search"]["run_to_convergence"] is None


@pytest.mark.timeout(900)
def test_bench_dumps_the_state_after_its_timed_steps(oracle, tmp_path):
    """--dump-outputs: the LLH, sumF and F the hot path returned after the last of the --steps timed steps, i.e. the
    oracle's state after the warm-up, settle and timed steps from the same seeded workload."""
    import bench
    out = str(tmp_path / "dump")
    d = _bench_dryrun("--steps", "3", "--no-cpu", "--no-init-a", "--no-line-search", "--dump-outputs", out)
    assert d["steps"] == 3 and d["dumped_outputs"]["F_rows"] == "all"
    assert sorted(os.listdir(out)) == ["F.npy", "llh.npy", "sumF.npy"]
    rp, col, F = bench.load_workload("rmat:150:500", 16)
    s, P = oracle.colsum(F), oracle.make_params(16)
    for _ in range(d["untimed_steps_before_timing"] + d["steps"]):
        r = oracle.step(rp, col, F, s, P)
        F, s = r.F, r.sumF
    llh, sumF, Fd = (np.load(os.path.join(out, f)) for f in ("llh.npy", "sumF.npy", "F.npy"))
    assert llh.dtype == sumF.dtype == Fd.dtype == np.float64 and Fd.shape == F.shape
    assert llh[0] == d["llh_end"] and abs(llh[0] - r.llh) <= 1e-10 * abs(r.llh)
    assert np.allclose(sumF, s, rtol=1e-11, atol=1e-9)
    assert np.abs(Fd - F).max() <= 1e-9 * np.abs(F).max()
