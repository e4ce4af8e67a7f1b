"""The stage of a frame denoised in parts, without a GPU: rt3_denoise_stage_words against the layout include/rt3cuda.h
documents (colour, guide and albedo planes, then one 64-bit fingerprint per row at an even word), the 0 for frames whose
stage rt3_frame_alloc cannot hold, and the resources of the stage kernel (cuobjdump on librt3cuda.so): no local memory,
no stack, at most 64 registers."""
import re
import shutil
import subprocess

import pytest

from rt3_b200 import abi

FRAME_ALLOC_MAX_WORDS = 2 ** 32 - 1


def layout_words(w, h):
    n = w * h
    planes = 4 * n + 4 * n + 3 * n              # rt3_dn_px, rt3_dn_guide (16 B each), 3 floats of albedo
    return planes + (planes & 1) + 2 * h          # fingerprints 8-byte aligned


@pytest.mark.parametrize("w,h", [(1, 1), (2, 2), (3, 1), (37, 21), (41, 23), (1200, 800), (3840, 2160), (65535, 2), (2, 65535)])
def test_stage_words_follow_the_layout(built, w, h):
    words = abi.denoise_stage_words(w, h)
    assert words == layout_words(w, h)
    assert (words - 2 * h) % 2 == 0                # the fingerprints start at an even word: 8-byte aligned in a cudaMalloc block


@pytest.mark.parametrize("w,h", [(0, 0), (0, 5), (5, 0)])
def test_empty_frames_have_no_stage(built, w, h):
    assert abi.denoise_stage_words(w, h) == 0


def test_oversize_frames_have_no_stage(built):
    # the largest square frame whose stage rt3_frame_alloc still takes, and the next one
    side = 19000
    assert layout_words(side, side) <= FRAME_ALLOC_MAX_WORDS < layout_words(side + 1000, side + 1000)
    assert abi.denoise_stage_words(side, side) == layout_words(side, side)
    assert abi.denoise_stage_words(side + 1000, side + 1000) == 0
    assert abi.denoise_stage_words(0xFFFFFFFF, 0xFFFFFFFF) == 0
    assert abi.denoise_stage_words(0xFFFFFFFF, 2) == 0
    # the boundary itself: the largest w x 2 frame that fits, then one more column
    w = (FRAME_ALLOC_MAX_WORDS - 4) // 22
    assert layout_words(w, 2) <= FRAME_ALLOC_MAX_WORDS < layout_words(w + 1, 2)
    assert abi.denoise_stage_words(w, 2) == layout_words(w, 2)
    assert abi.denoise_stage_words(w + 1, 2) == 0


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_stage_kernel_keeps_to_registers(built):
    text = subprocess.run(["cuobjdump", "-res-usage", abi.CORE_LIB_PATH], check=True, capture_output=True, text=True).stdout
    found = [(m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in
             re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", text) if "denoise_stage_kernel" in m.group(1)]
    assert len(found) == 1, found
    name, reg, stack, local = found[0]
    assert local == 0 and stack == 0, f"{name}: {local} bytes of local memory, {stack} bytes of stack"
    assert reg <= 64, f"{name}: {reg} registers"
