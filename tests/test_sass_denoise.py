"""The denoiser's kernels (rt3_denoise) keep to registers (no GPU needed: cuobjdump on librt3cuda.so): no local memory in any
of them, no stack but the division slow path's, and the register counts ptxas reports leave every 256-thread CTA room for full occupancy (at most 64 per thread,
65 536 / (256 * 4)). The existing kernels were left unchanged by them; DESIGN.md 3.8 says how that was checked."""
import re
import shutil
import subprocess

import pytest

from rt3_b200 import abi

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")

KERNELS = ["denoise_prepare_kernel", "denoise_variance_kernel", "denoise_atrous_kernelILb0E", "denoise_atrous_kernelILb1E"]


@pytest.fixture(scope="module")
def resources(built):
    text = subprocess.run(["cuobjdump", "-res-usage", abi.CORE_LIB_PATH], check=True, capture_output=True, text=True).stdout
    return [(m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in
            re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", text)]


@pytest.mark.parametrize("needle", KERNELS)
def test_no_local_memory_and_few_registers(resources, needle):
    found = [r for r in resources if needle in r[0]]
    assert len(found) == 1, found
    name, reg, stack, local = found[0]
    assert local == 0, f"{name}: {local} bytes of local memory"
    # the last pass's 16-byte stack frame is the register save of the IEEE division's slow-path subroutine, which runs only
    # for operands the fast path cannot take (FCHK); the other kernels have none
    assert stack <= (16 if "ILb1E" in name else 0), f"{name}: {stack} bytes of stack"
    assert reg <= 64, f"{name}: {reg} registers"
