"""The parts of bench.py that run on the host cores only — the reference arm and its JSON contract, the output dump,
the argument checks — are checked here."""
import json
import os
import subprocess
import sys

from conftest import REPO


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "edges/sec in F-gradient step" and d["unit"] == "edges/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["config"]["workload"].startswith("com-amazon K=200") and d["config"]["nnz_directed"] == 1851744
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert 1e4 < d["value"] < 1e9 and abs(d["value"] - 1851744 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=REPO, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_uses_all_cores_under_torchrun_env():
    """torchrun exports OMP_NUM_THREADS=1; the reference arm must time the CPU restatement on the box's cores anyway,
    with the same steps / warm-up it was asked for and the same config keys as the GPU arm."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1",
                          "--config", "enron50"], capture_output=True, text=True, timeout=600, cwd=REPO, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 2
    assert set(d["config"]) == {"workload", "graph", "k", "n", "nnz_directed", "edges_undirected", "f0", "f_layout"}
    assert d["config"]["graph"] == "email-enron" and d["config"]["k"] == 50


def test_dump_outputs_samples_a_large_F_within_the_budget(tmp_path):
    """An F too large for the dump is replaced by the same seeded sample of its rows in every run, the whole dump < 64 MB."""
    import numpy as np
    import scipy.sparse as sps

    import bench

    n, k = 20000, 1000
    m = sps.random(n, k, density=0.01, format="csr", random_state=np.random.default_rng(5))

    class Engine:
        K = k
        sumF = np.asarray(m.sum(axis=0)).ravel()

        def F_csr(self):
            return m.indptr.astype(np.int64), m.indices.astype(np.int32), m.data

    a = bench.dump_outputs(str(tmp_path / "a"), Engine(), -1.5)
    bench.dump_outputs(str(tmp_path / "b"), Engine(), -1.5)
    rows = np.sort(np.random.default_rng(0).choice(n, bench.DUMP_F_BYTES // (8 * k), replace=False))
    F = np.load(tmp_path / "a" / "F.npy")
    assert a["F_rows"].startswith(f"{len(rows)} of {n} rows") and np.array_equal(F, m[rows].toarray())
    assert np.array_equal(F, np.load(tmp_path / "b" / "F.npy"))
    assert np.load(tmp_path / "a" / "llh.npy").tolist() == [-1.5]
    assert np.array_equal(np.load(tmp_path / "a" / "sumF.npy"), Engine.sumF)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in a["files"]) < 64 << 20


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=REPO)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr
