"""rt3_denoise_staged_temporal's kernel keeps to registers like the other denoise kernels (tests/test_sass_denoise.py), no
GPU needed: cuobjdump on librt3cuda.so shows no local memory, no stack and at most 64 registers per thread (full occupancy
of its 256-thread CTAs, 65 536 / (256 * 4))."""
import re
import shutil
import subprocess

import pytest

from rt3_b200 import abi

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")

KERNEL = "denoise_staged_temporal_kernel"


def test_no_local_memory_no_stack_and_few_registers(built):
    text = subprocess.run(["cuobjdump", "-res-usage", abi.CORE_LIB_PATH], check=True, capture_output=True, text=True).stdout
    found = [(m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in
             re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", text) if m.group(1).startswith(f"_Z{len(KERNEL)}{KERNEL}")]
    assert len(found) == 1, found
    name, reg, stack, local = found[0]
    assert local == 0, f"{name}: {local} bytes of local memory"
    assert stack == 0, f"{name}: {stack} bytes of stack"
    assert reg <= 64, f"{name}: {reg} registers"
