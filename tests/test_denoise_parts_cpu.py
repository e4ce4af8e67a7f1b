"""The stage of a frame denoised in parts, without a GPU: rt3_denoise_stage_words against the layout include/rt3cuda.h
documents (colour, guide and albedo planes, then one 64-bit fingerprint per row at an even word) and the 0 for frames whose
stage rt3_frame_alloc cannot hold. The stage kernel's resources are checked in tests/test_sass_denoise.py."""
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

