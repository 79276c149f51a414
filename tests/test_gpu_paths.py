"""The two ways kCull's work can be organised (garden_b200/csrc/cull.cu) must give the same bits: the FUSED kernel (chains found
among the pool's own survivors) and the SPLIT path (world matrices per surviving transform, then kClassify per pool). The
library picks per pool at link time; here every parity suite that is quick is re-run with the choice forced either way
(GSP_SPLIT is read once per process, hence the subprocesses), plus the prepass and the box-view shortcut switched off."""
import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
QUICK = ["tests/test_gpu_fuzz.py", "tests/test_gpu_golden.py", "tests/test_gpu_next.py", "tests/test_gpu_hostpath.py",
         "tests/test_gpu_parity.py", "tests/test_gpu_shapes.py"]


@pytest.mark.parametrize("env", [{"GSP_SPLIT": "1"}, {"GSP_SPLIT": "0"}, {"GSP_PREPASS": "0"}, {"GSP_BOXGROUP": "0"},
                                 {"GSP_SPLIT": "1", "GSP_PREPASS": "0"}],
                         ids=["split", "fused", "no-prepass", "no-boxgroup", "split-no-prepass"])
def test_forced_paths_give_the_same_bits(sceneprep_lib, oracle_built, env):
    res = subprocess.run([sys.executable, "-m", "pytest", *QUICK, "-m", "gpu", "-x", "-q", "-k", "not full_size and not shortcuts"],
                         cwd=ROOT, env={**os.environ, **env}, capture_output=True, text=True, timeout=1500)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-1000:]
