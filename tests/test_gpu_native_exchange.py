"""The multi-GPU path driven purely through the C ABI by a C++ program (tests/native/exchange_two_ranks.cpp): two GPUs, one
process, one thread per GPU, NCCL inside the library, no Python in the data path. Needs two devices: marked `multigpu`, which
tests/conftest.py skips on a box with fewer than two GPUs (log of a two-GPU run under profiles/)."""
import os
import shutil
import subprocess
from pathlib import Path

import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]
ROOT = Path(__file__).resolve().parent.parent


def _device_count() -> int:
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return sum(1 for ln in out.splitlines() if ln.startswith("GPU "))
    except Exception:
        return 0


@pytest.mark.parametrize("protocol", ["alltoall", "allgather"])
def test_two_ranks_without_python(sceneprep_lib, tmp_path, protocol):
    if _device_count() < 2:
        pytest.skip("needs two GPUs")
    if shutil.which("g++") is None:
        pytest.skip("g++ not on PATH")
    exe = tmp_path / "exchange_two_ranks"
    res = subprocess.run(["g++", "-std=c++17", "-O2", "-I", str(ROOT / "include"), str(ROOT / "tests/native/exchange_two_ranks.cpp"),
                          "-L", str(sceneprep_lib.parent), "-lgarden_sceneprep", "-lpthread", "-o", str(exe)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    env = {**os.environ, "LD_LIBRARY_PATH": f"{sceneprep_lib.parent}:{os.environ.get('LD_LIBRARY_PATH', '')}", "GSP_EXCHANGE": protocol}
    run = subprocess.run([str(exe), "2"], capture_output=True, text=True, env=env, timeout=600)
    assert run.returncode == 0, run.stdout[-1000:] + run.stderr[-2000:]
    assert "ok" in run.stdout and protocol in run.stdout
