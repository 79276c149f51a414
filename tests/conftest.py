import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "multigpu: needs at least two CUDA devices (skipped where fewer exist)")


def _device_usable() -> bool:
    """True when gsp_create(0) succeeds, i.e. an sm_100 device is usable by the product library."""
    try:
        import ctypes as C
        from garden_b200.build import build_library
        build_library()
        from garden_b200.binding import load_library
        lib = load_library()
        h = C.c_void_p()
        if lib.gsp_create(0, C.byref(h)) != 0:
            return False
        lib.gsp_destroy(h)
        return True
    except Exception:
        return False


def _gpu_count() -> int:
    try:
        import subprocess
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return sum(1 for ln in out.splitlines() if ln.startswith("GPU "))
    except Exception:
        return 0


def pytest_collection_modifyitems(config, items):
    """(1) `multigpu` tests are skipped where fewer than two GPUs exist: they stay in the report of a single-GPU run. (2) A
    plain `pytest tests` on a box without a usable sm_100 device skips the gpu-marked tests instead of failing them
    (tests/test_abi.py::test_no_cpu_fallback stays the one place that asserts the loud failure). With `-m gpu` nothing else
    is skipped: a missing device must fail there, not pass silently."""
    multi = [it for it in items if it.get_closest_marker("multigpu")]
    if multi and _gpu_count() < 2:
        for it in multi:
            it.add_marker(pytest.mark.skip(reason="needs at least two CUDA devices"))
    markexpr = config.getoption("-m", default="") or ""
    if "gpu" in markexpr and "not gpu" not in markexpr:
        return
    gpu_items = [it for it in items if it.get_closest_marker("gpu")]
    if not gpu_items or _device_usable():
        return
    skip = pytest.mark.skip(reason="no usable sm_100 CUDA device (the scene-preparation path has no CPU fallback)")
    for it in gpu_items:
        it.add_marker(skip)


@pytest.fixture(scope="session")
def oracle_built():
    from reflib import build_oracle
    return build_oracle()


@pytest.fixture(scope="session")
def sceneprep_lib():
    """The product library; (re)built in-tree when sources are newer (nvcc cross-compiles without a GPU)."""
    from garden_b200.build import build_library
    return build_library()
