"""rt3_denoise on the GPU against the float64 reference tests/denoise_ref.py, on the radiance and AOVs of GPU renders: the
tolerance, 8-bit frame rule, convex-hull bound and mutation rule of tests/test_denoise_reference.py, applied to the kernels'
own output. tests/test_gpu_denoise.py pins the kernels to the CPU restatement bit for bit; both share include/rt3_denoise.h,
and this file is what checks that arithmetic on the device. The kernels read the context's accumulators and AOVs, so every
case starts from a render.

Rendered inputs, unlike the synthetic ones, are near-constant in many 7x7 windows once demodulated: the gradient sky divided
by its own colour (constant to about 5e-4), and pixels whose window the geometry weights reduce to the centre. There the
variance E[L^2] - E[L]^2 cancels by more than 2^12 and its float32 value has lost most of its bits, so the luminance stop
is ill-conditioned: the kernels (and the restatement, on the same inputs) were measured up to 2.4e-2 from the reference on
such pixels. Those pixels, and every pixel that later reads them, are held to the hull bound only (ill_conditioned()); the
mutation test compares every pixel. Also: a progressive (RT3_FLAG_ACCUMULATE) render denoises exactly like a one-shot render of all
its samples."""
import numpy as np
import pytest

import denoise_ref as ref
import fullsize as fs
from rt3_b200 import abi, scenes
from test_denoise_reference import compare, demodulated, rel_error, tau
from test_gpu_path_aovs import scene_of

pytestmark = pytest.mark.gpu

# (width, height): partial 32x8 tiles in x, in y and in both, one exact tile, and frames thinner than a pass's step
SIZES = [(33, 9), (32, 8), (31, 7), (257, 3), (3, 257)]


def camera(w, h, lens):
    cam = abi.reference_camera(w, h)
    if lens:
        cam.lens_radius = 0.08
        cam.lens_u[:] = [1, 0, 0]
        cam.lens_v[:] = [0, 1, 0]
    return cam


def render(ctx, cam, w, h, spp=8, aov_spp=4, flags=0, depth=5, seed=3):
    """Render, AOVs, read_radiance: the inputs rt3_denoise reads, as (radiance, albedo, normal, depth) arrays."""
    ctx.render(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=depth, seed=seed, flags=flags))
    aov = ctx.render_path_aovs(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=aov_spp, max_depth=depth, seed=seed, flags=flags))
    return ctx.read_radiance(w, h), aov["albedo"], aov["normal"], aov["hit_t"]


def gpu_passes(ctx, inp, **dn):
    """rt3_denoise at 1..iterations: the demodulated colour after every pass, and the last (frame, rgb)."""
    h, w = inp[3].shape
    passes = []
    for i in range(1, dn.get("iterations", 5) + 1):
        frame, out = ctx.denoise(w, h, **{**dn, "iterations": i})
        passes.append(demodulated(out, inp[1]))
    return passes, frame, out


def check(ctx, inp, what, flags=0, **dn):
    passes, frame, _ = gpu_passes(ctx, inp, **dn)
    return compare(inp, passes, frame, what, flags, skip_ill=True, **dn)


@pytest.mark.parametrize("flag", ["none", "bvh"])
@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("name", ["c1", "cloud", "mesh"])
def test_against_the_reference(gpu_ctx, name, lens, flag):
    """Every pass of 8 (so the results of 1 to 8 iterations) at every size of SIZES."""
    gpu_ctx.upload(scene_of(name))
    flags = abi.FLAG_BVH if flag == "bvh" else 0
    for w, h in SIZES:
        check(gpu_ctx, render(gpu_ctx, camera(w, h, lens), w, h, flags=flags), f"{name} {w}x{h}", flags, iterations=8)


@pytest.mark.parametrize("dn", [dict(sigma_luminance=0.5, sigma_normal=7.0, sigma_depth=0.05), dict(iterations=8, sigma_luminance=40.0, sigma_normal=1.0, sigma_depth=10.0)])
def test_non_default_parameters(gpu_ctx, dn):
    scene, cam = scenes.rtiow_four_spheres(61, 45)
    gpu_ctx.upload(scene)
    check(gpu_ctx, render(gpu_ctx, cam, 61, 45, 4, 2), str(dn), **dn)


def test_c2_full_size(gpu_ctx):
    """C2 at 1200x800, 16 samples and 16 AOV samples, 5 iterations."""
    c = fs.CONFIGS["c2"]
    w, h = c["w"], c["h"]
    scene, cam = c["scene"](w, h)
    gpu_ctx.upload(scene)
    check(gpu_ctx, render(gpu_ctx, cam, w, h, 16, 16, c["flags"], c["depth"], seed=1), "C2", c["flags"], iterations=5)


@pytest.mark.parametrize("mutation", list(ref.MUTATIONS))
def test_mutation_is_detected(gpu_ctx, mutation):
    """Each mutation of the reference is more than 10 tau from the kernels' output on C1 at 61x45 (5 iterations, the
    defaults). Measured on a B200: 0.31 (reach_one) to inf (no_centre_in_sum: 0 / 0 where no other tap has weight)."""
    scene, cam = scenes.rtiow_four_spheres(61, 45)
    gpu_ctx.upload(scene)
    inp = render(gpu_ctx, cam, 61, 45, 8, 4)
    passes, _, _ = gpu_passes(gpu_ctx, inp, iterations=5)
    res = ref.denoise(*inp, mutation=mutation, iterations=5)
    err = max(rel_error(a, b) for a, b in zip(passes, res["passes"]))
    assert err > 10 * tau(), f"{mutation}: {err:.3g}"
    print(f"{mutation}: {err:.3g}")


def test_progressive_render_denoises_like_one_shot(gpu_ctx):
    """k RT3_FLAG_ACCUMULATE passes of n samples, then rt3_denoise, equal the denoise of one render of k n samples, frame and
    rgb bit for bit: the radiance is the accumulator over the whole sample count (resolve_spp), not over the last pass's."""
    w, h, k, n = 61, 45, 3, 4
    scene, cam = scenes.rtiow_four_spheres(w, h)
    gpu_ctx.upload(scene)
    gpu_ctx.render_path_aovs(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=4, max_depth=8, seed=5))
    for i in range(k):
        gpu_ctx.render(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=n, max_depth=8, seed=5, first_sample=i * n,
                                            flags=abi.FLAG_ACCUMULATE if i else 0))
    progressive = gpu_ctx.denoise(w, h)
    gpu_ctx.render(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=k * n, max_depth=8, seed=5))
    once = gpu_ctx.denoise(w, h)
    assert np.array_equal(progressive[0], once[0])
    assert np.array_equal(progressive[1].view(np.uint32), once[1].view(np.uint32))
