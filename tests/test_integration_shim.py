"""The reference-side binding shown in INTEGRATION.md is real code: both C++ blocks are extracted and compiled
(-fsyntax-only) against the reference's own headers and include/garden_sceneprep.h. Needs a checkout of the reference
(github.com/cfnptr/garden) named by the GARDEN_REFERENCE environment variable; skipped without one."""
import os
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
REF = Path(os.environ["GARDEN_REFERENCE"]) if os.environ.get("GARDEN_REFERENCE") else None
GEN = ROOT / "oracle" / "_ref" / "gen"

# os.path.isfile: False (not PermissionError) where the path lies in a directory this user may not read
pytestmark = pytest.mark.skipif(REF is None or not os.path.isfile(REF / "include" / "garden" / "system" / "render" / "mesh.hpp"),
                                reason="GARDEN_REFERENCE does not name a checkout of the reference")


def test_integration_shim_compiles_against_reference_headers(tmp_path):
    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), f"REF={REF}", "_ref/gen/garden/defines.hpp"], check=True)
    md = (ROOT / "INTEGRATION.md").read_text()
    blocks = re.findall(r"```cpp\n(.*?)```", md, re.S)
    assert len(blocks) >= 2, "INTEGRATION.md should hold the shim and the 8f callers"
    src = tmp_path / "mesh_b200.cpp"
    src.write_text("\n".join(blocks))
    inc = [GEN, REF / "include", REF / "shaders", REF / "libraries/math/include", REF / "libraries/ecsm/include",
           REF / "libraries/ecsm/libraries/robin-map/include", REF / "libraries/logy/include", REF / "libraries/logy/wrappers/cpp",
           REF / "libraries/logy/libraries/mpio/include", REF / "libraries/logy/libraries/mpio/wrappers/cpp",
           REF / "libraries/logy/libraries/mpmt/include", REF / "libraries/logy/libraries/mpmt/wrappers/cpp",
           REF / "libraries/json/include", REF / "libraries/pack/include", REF / "libraries/pack/wrappers/cpp", ROOT / "include"]
    # -fno-access-control stands in for the `friend struct B200Prep;` line a maintainer adds to MeshRenderSystem
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-fno-access-control", "-DNDEBUG", "-march=haswell",
           *[f"-I{p}" for p in inc], str(src)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
