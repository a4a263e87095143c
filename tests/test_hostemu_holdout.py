"""The masked step and the held-out LLH on the CPU: a selection of the `-m gpu` tests of tests/test_gpu_holdout.py, run in
a child pytest against the host-emulation build of the C API (tests/emu/build_hostemu.sh, see tests/test_hostemu_sparse.py).
Covers the kHO instantiation of tile_step_kernel (general path with held-out lists, no tiles, no bounds), nodes with only
held-out pairs, the uset mask, the held-out LLH kernel and its fixed-order sum, bit-identical reruns, clearing, the input
checks of bigclam_set_holdout, the C++ wrappers and the device-side loop."""
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SELECTION = ("(random_graphs and (31 or 65)) or uset or only_held_out or bit_identical or clearing or input_errors or "
             "holdout_llh or cpp_wrappers or run_follows")


@pytest.mark.timeout(1800)
def test_masked_step_under_host_emulation():
    env = dict(os.environ, BIGCLAM_HOSTEMU="1")
    env.pop("BIGCLAM_HOSTEMU_NOBUILD", None)
    cmd = [sys.executable, "-m", "pytest", os.path.join(REPO, "tests", "test_gpu_holdout.py"), "-m", "gpu", "-q", "-x",
           "-p", "no:cacheprovider", "-k", SELECTION]
    r = subprocess.run(cmd, cwd=REPO, env=env, capture_output=True, text=True, timeout=1700)
    tail = "\n".join((r.stdout + r.stderr).splitlines()[-25:])
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail
