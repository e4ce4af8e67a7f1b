"""The denoiser (rt3_denoise) on the CPU: the restatement tests/denoise_oracle.c, which runs the filter arithmetic of
include/rt3_denoise.h as the kernels do, on synthetic inputs whose results can be checked by hand; the quality bar on C1
with the oracle's path tracer; parameter validation and the ABI struct's layout. No GPU needed."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import denoise_lib as dl
import oraclelib as ol
import path_aov_lib as pal
from rt3_b200 import abi, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INF = np.float32(np.inf)


def inputs(h, w, colour=0.3, albedo=0.6, normal=(0.0, 0.0, 1.0), depth=2.0):
    return (np.full((h, w, 3), colour, np.float32), np.full((h, w, 3), albedo, np.float32), np.broadcast_to(np.float32(normal), (h, w, 3)).copy(),
            np.full((h, w), depth, np.float32))


def ulp_distance(a, b):
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


@pytest.mark.parametrize("colour,albedo", [(0.3, 0.6), (0.25, 0.5), (0.7, 0.9), (0.05, 0.0)])
def test_constant_inputs_come_back(colour, albedo):
    rgb, a, n, z = inputs(23, 37, colour, albedo)
    frame, out = dl.oracle_denoise(rgb, a, n, z)
    assert ulp_distance(out, rgb).max() <= 2
    gamma = ol.resolve_8bit(rgb)
    assert np.array_equal(ol.unpack_rgb(frame), gamma)


def test_constant_sky_comes_back():
    rgb, a, n, z = inputs(16, 16, 0.8, 0.8, normal=(0, 0, 0), depth=np.inf)
    _, out = dl.oracle_denoise(rgb, a, n, z)
    assert ulp_distance(out, rgb).max() <= 2


def noisy(h, w, seed=1):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.0, 1.0, (h, w, 3)).astype(np.float32)


def test_orthogonal_normals_separate_the_halves():
    """Left half faces +z, right half +x: the normal term of every tap across the split is max(0, 0)^128 = 0, so nothing on
    the right reaches the left, at any step."""
    h, w = 24, 40
    rgb, a, n, z = inputs(h, w)
    rgb = noisy(h, w)
    n[:, w // 2:] = (1, 0, 0)
    left = dl.oracle_denoise(rgb, a, n, z)
    rgb2 = rgb.copy()
    rgb2[:, w // 2:] = noisy(h, w - w // 2, seed=2) * np.float32(5)
    right = dl.oracle_denoise(rgb2, a, n, z)
    assert np.array_equal(left[1][:, :w // 2].view(np.uint32), right[1][:, :w // 2].view(np.uint32))
    assert np.array_equal(left[0][:, :w // 2], right[0][:, :w // 2])
    assert not np.array_equal(left[1][:, w // 2:], right[1][:, w // 2:])


def test_misses_and_hits_do_not_mix():
    h, w = 24, 40
    rgb, a, n, z = inputs(h, w)
    rgb = noisy(h, w)
    z[:, :w // 2] = INF
    n[:, :w // 2] = 0
    base = dl.oracle_denoise(rgb, a, n, z)
    for side, other in ((slice(w // 2, None), slice(None, w // 2)), (slice(None, w // 2), slice(w // 2, None))):
        rgb2 = rgb.copy()
        rgb2[:, side] = rgb2[:, side] * np.float32(3) + np.float32(0.5)
        pert = dl.oracle_denoise(rgb2, a, n, z)
        assert np.array_equal(base[1][:, other].view(np.uint32), pert[1][:, other].view(np.uint32))


def test_demodulation_keeps_an_albedo_checkerboard():
    """Constant irradiance E times a checkerboard albedo: the demodulated image is E everywhere, so the filter returns
    E * albedo again and the checkerboard survives, where a filter of the radiance itself would blur it."""
    h, w = 32, 48
    yy, xx = np.mgrid[:h, :w]
    board = np.where(((yy // 2) + (xx // 2)) % 2 == 0, np.float32(0.9), np.float32(0.1)).astype(np.float32)
    a = np.repeat(board[..., None], 3, axis=2)
    irradiance = np.float32(0.5)
    rgb = a * irradiance
    _, n, z = inputs(h, w)[1:]
    frame, out = dl.oracle_denoise(rgb, a, n, z)
    assert np.abs(out - rgb).max() <= 1e-6
    assert np.array_equal(ol.unpack_rgb(frame), ol.resolve_8bit(rgb))


@pytest.mark.parametrize("shape", [(1, 1), (1, 64), (64, 1), (2, 3)])
@pytest.mark.parametrize("iterations", [1, 5, 8])
def test_thin_images_give_no_nan(shape, iterations):
    h, w = shape
    rgb, a, n, z = inputs(h, w)
    rgb = noisy(h, w)
    z[..., ::2] = INF
    frame, out = dl.oracle_denoise(rgb, a, n, z, iterations=iterations)
    assert np.isfinite(out).all()
    assert (out >= 0).all()


def test_no_gamma_resolves_the_linear_value():
    rgb, a, n, z = inputs(8, 8, 0.25, 0.5)
    frame, out = dl.oracle_denoise(rgb, a, n, z, flags=abi.FLAG_NO_GAMMA)
    assert np.array_equal(ol.unpack_rgb(frame), ol.resolve_8bit(out, gamma=False))


def test_one_pass_on_two_pixels_by_hand():
    """One pass over a 1x2 image against the formula evaluated in float64: checks the header's exp(-x), the variance estimate
    and the luminance term together to a relative 2e-6."""
    rgb, a, n, z = inputs(1, 2)
    # a 1x2 image at one pass: the right pixel's output is (9/64 c1 + (1/4 * 3/8) w c0) / (9/64 + 3/32 w), w = exp(-x_l) with
    # x_l = |L1 - L0| / (sigma_l * sqrt(g) + 1e-10); the variance g is that of the 7x7 estimate, here 0.25 (L 0 and 1)
    for d in (0.0, 0.1, 0.5, 1.0, 2.0):
        rgb = np.zeros((1, 2, 3), np.float32)
        rgb[0, 1] = np.float32(d)
        a[:] = 1
        _, out = dl.oracle_denoise(rgb, a, n, z, iterations=1, sigma_luminance=1.0)
        lum = np.float64(0.2126 + 0.7152 + 0.0722) * d
        var = 0.25 * lum * lum  # E[L^2] - E[L]^2 over the two pixels, equal weights
        x = lum / (np.sqrt(var) + 1e-10) if d else 0.0
        w = np.exp(-x)
        want = (9 / 64 * d) / (9 / 64 + 3 / 32 * w)
        assert out[0, 1, 0] == pytest.approx(want, rel=2e-6, abs=1e-12)


@pytest.mark.parametrize("bad", [dict(iterations=0), dict(iterations=9), dict(sigma_luminance=0.0), dict(sigma_luminance=-1.0),
                                 dict(sigma_luminance=float("inf")), dict(sigma_luminance=float("nan")), dict(sigma_depth=0.0),
                                 dict(sigma_depth=float("inf")), dict(sigma_normal=0.0), dict(sigma_normal=0.5), dict(sigma_normal=127.5),
                                 dict(sigma_normal=1025.0), dict(sigma_normal=float("nan"))])
def test_parameter_validation(bad):
    assert dl.check_params(**bad) is not None


@pytest.mark.parametrize("good", [dict(), dict(iterations=1), dict(iterations=8), dict(sigma_normal=1.0), dict(sigma_normal=1024.0),
                                  dict(sigma_luminance=1e-3, sigma_depth=1e6)])
def test_valid_parameters(good):
    assert dl.check_params(**good) is None


def test_params_layout_matches_the_header():
    text = open(os.path.join(ROOT, "include", "rt3cuda.h")).read()
    body = re.search(r"typedef struct rt3_denoise_params \{(.*?)\} rt3_denoise_params;", text, re.S).group(1)
    fields = []
    for line in body.splitlines():
        m = re.match(r"\s*(uint32_t|float)\s+([\w, ]+);", line)
        if m:
            fields += [(name.strip(), m.group(1)) for name in m.group(2).split(",")]
    ctypes_of = {"uint32_t": C.c_uint32, "float": C.c_float}
    assert [(f, ctypes_of[t]) for f, t in fields] == abi.DenoiseParams._fields_
    assert C.sizeof(abi.DenoiseParams) == 24
    assert "rt3_denoise" in abi.EXPORTED_SYMBOLS


QW, QH = 200, 113


@pytest.fixture(scope="module")
def c1_quality():
    """C1 at 200x113 with the oracle: 16 and 64 spp (seed 1), a 4096-spp reference (another seed), the 16-sample AOVs."""
    scene, cam = scenes.rtiow_four_spheres(QW, QH)

    def render(spp, seed):
        p = abi.make_params(QW, QH, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=50, seed=seed)
        frame, acc, _ = ol.oracle_pathtrace(scene, cam, p, want_accum=True)
        return frame, (acc.astype(np.float64) / (spp * 16777216.0)).astype(np.float32)

    f16, r16 = render(16, 1)
    f64, _ = render(64, 1)
    ref, _ = render(4096, 77)
    aov = pal.oracle_path_aovs(scene, cam, abi.make_params(QW, QH, mode=abi.MODE_PATHTRACE, spp=16, max_depth=50, seed=1))
    den, _ = dl.oracle_denoise(r16, aov["albedo"], aov["normal"], aov["hit_t"])
    refl = ol.unpack_rgb(ref)
    return {k: ol.psnr_levels(ol.unpack_rgb(f), refl) for k, f in (("raw16", f16), ("raw64", f64), ("denoised16", den))}


def test_denoising_beats_the_raw_16_samples(c1_quality):
    q = c1_quality
    assert q["denoised16"] > q["raw16"] + 5.0, q


@pytest.mark.xfail(strict=True, reason="measured with the default parameters: 35.46 dB for 16 spp denoised against 35.74 dB for 64 raw "
                                      "spp (DESIGN.md 3.8); the bar is kept")
def test_denoising_is_worth_four_times_the_samples(c1_quality):
    q = c1_quality
    assert q["denoised16"] > q["raw64"], q
