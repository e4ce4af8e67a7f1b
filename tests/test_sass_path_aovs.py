"""The AOV kernel of the path tracer's primary rays keeps the sweep's code generation (no GPU needed: cuobjdump on
librt3cuda.so): packed FMAs with uniform operands out of the constant bank, bulk copies for streamed scenes, and no local
memory in any instantiation. The existing kernels were left unchanged by it; DESIGN.md 3.7 says how that was checked."""
import re
import shutil
import subprocess

import pytest

from rt3_b200 import abi

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")

# path_aov_kernel<RESIDENT, SPHERES_ONLY, ACCEL>
CONSTANT_BANK = ["path_aov_kernelILb1ELb1ELb0E", "path_aov_kernelILb1ELb0ELb0E"]
STREAMED = ["path_aov_kernelILb0ELb1ELb0E", "path_aov_kernelILb0ELb0ELb0E"]
HIERARCHY = ["path_aov_kernelILb1ELb0ELb1E"]


@pytest.fixture(scope="module")
def sass(built):
    text = subprocess.run(["cuobjdump", "-sass", abi.CORE_LIB_PATH], check=True, capture_output=True, text=True).stdout
    kernels = {}
    for block in text.split("Function : ")[1:]:
        name, _, body = block.partition("\n")
        kernels[name.strip()] = re.findall(r"^\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", body, flags=re.M)
    return kernels


def ops_of(sass, needle):
    names = [n for n in sass if needle in n]
    assert len(names) == 1, names
    return sass[names[0]]


@pytest.mark.parametrize("needle", CONSTANT_BANK)
def test_constant_bank_instantiation_sweeps_with_packed_fma_and_uniform_loads(sass, needle):
    ops = ops_of(sass, needle)
    assert sum(op.startswith("FFMA2") for op in ops) >= 96
    assert sum(op == "LDCU.64" for op in ops) >= 48, "the records are no longer read through uniform registers"
    assert any(op.startswith("RED") and "64" in op for op in ops), "no 64-bit reduction for the fixed-point sums"


@pytest.mark.parametrize("needle", STREAMED)
def test_streamed_instantiation_stages_tiles_with_bulk_copies(sass, needle):
    ops = ops_of(sass, needle)
    assert sum(op.startswith("UBLKCP") for op in ops) >= 2
    assert sum(op.startswith("FFMA2") for op in ops) >= 96


@pytest.mark.parametrize("needle", CONSTANT_BANK + STREAMED + HIERARCHY + ["path_aov_resolve_kernel"])
def test_no_local_memory(built, needle):
    text = subprocess.run(["cuobjdump", "-res-usage", abi.CORE_LIB_PATH], check=True, capture_output=True, text=True).stdout
    found = [(m.group(1), int(m.group(2))) for m in re.finditer(r"Function (\S+):\s*\n\s*REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:(\d+)", text) if needle in m.group(1)]
    assert len(found) == 1, found
    assert found[0][1] == 0, f"{found[0][0]}: {found[0][1]} bytes of local memory"
