"""The projection kernels' shared-memory matrix products run on the fp64 tensor cores (DESIGN.md section 4): the
object of tce_proj.cu contains DMMA and no tensor-core instruction of the fp16 / tf32 paths.  Checked on the object
file of the in-tree build (cuobjdump, no GPU needed)."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_projection_products_are_dmma_and_nothing_else_is_on_the_tensor_cores():
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "tce_rl_b200", "build", "tce_proj.o")
    if not os.path.exists(tool) or not os.path.exists(obj):
        pytest.skip("cuobjdump or the object files of the in-tree build are not here")
    sass = subprocess.run([tool, "-sass", obj], capture_output=True, text=True, check=True).stdout
    opcodes = set(re.findall(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.x]*)", sass))
    mma = {op for op in opcodes if "MMA" in op}
    assert "DMMA.8x8x4" in mma
    assert mma == {"DMMA.8x8x4"}, mma            # no HMMA, no UTC*MMA (tcgen05)
