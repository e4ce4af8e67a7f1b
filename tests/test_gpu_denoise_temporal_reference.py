"""rt3_denoise_temporal and rt3_denoise_staged_temporal on the GPU against the float64 reference of the whole call,
``denoise_temporal_ref.temporal_denoise``, on GPU renders: the tolerance, 8-bit frame rule, hull bound and exclusions of
tests/test_denoise_temporal_reference.py applied to the kernels' own output at every frame of 6-frame sequences (a new seed
per frame, so that frames 4-6 take the moments' variance). tests/test_gpu_denoise_temporal.py pins the kernels to the CPU
restatement bit for bit; both share include/rt3_denoise.h, and this file is what checks that arithmetic on the device.

The history lives on the context, so every pass of every frame comes from replaying the sequence (``reset`` on its first
frame) once per iteration count. The reference's rays are the restatement's ``primary_ray`` (denoise_lib.primary_rays),
which the path-AOV tests pin bit for bit to the GPU's ``start_path``. The hull of the first pass is taken around the
restatement's accumulated colour, which equals the kernels' (tests/test_gpu_denoise_temporal.py). Each test prints its
worst errors and the pixel-frames held to the hull."""
import numpy as np
import pytest

import denoise_lib as dl
import denoise_temporal_ref as tref
from rt3_b200 import abi, scenes
from test_denoise_temporal_reference import ITERATIONS, Held, check_frame
from test_gpu_denoise_parts import Stage
from test_gpu_denoise_parts_temporal import parts_ctx, stage_frame  # noqa: F401  (parts_ctx is a fixture)
from test_gpu_denoise_temporal import cam_of, motion
from test_gpu_path_aovs import scene_of

pytestmark = pytest.mark.gpu

f32 = np.float32
FRAMES = 6
# (width, height): partial 32x8 tiles in x and in y, frames thinner than a pass's step, and one with room for every pass
SIZES = [(33, 9), (31, 7), (257, 3), (3, 257), (61, 45)]


def camera(kind, w, h, i, lens, base=None):
    """motion()'s cameras, and a `dolly` of 0.05 per frame along the view direction."""
    if kind != "dolly":
        return motion(kind, w, h, i, lens, base=base)
    base = base or abi.reference_camera(w, h)
    o, hor, ver, llc = (np.array(getattr(base, k)[:], f32) for k in ("origin", "horizontal", "vertical", "lower_left_corner"))
    shift = np.array([0.0, 0.0, -0.05 * i], f32)
    return cam_of(o + shift, hor, ver, llc + shift, lens)


def render(ctx, cam, w, h, seed, flags=0, spp=4, aov_spp=2, depth=5):
    """Render, AOVs, read_radiance: ((radiance, albedo, normal, depth), the AOV call's params)."""
    ctx.render(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=depth, seed=seed, flags=flags))
    a = abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=aov_spp, max_depth=depth, seed=seed, flags=flags)
    aov = ctx.render_path_aovs(cam, a)
    return (ctx.read_radiance(w, h), aov["albedo"], aov["normal"], aov["hit_t"]), a


class Totals(Held):
    def report(self, what):
        super().report(what)
        # rendered frames are mostly ill-conditioned (DESIGN.md 3.8, 3.9): the first pass must still compare some pixels
        assert self.share()[0] < 1.0, "every pixel-frame of the first pass held to the hull"


def check_sequence(cams, w, h, seed, run_frame, what, totals, mutation=None):
    """Frames `cams` (seeds seed, seed + 1, ...). ``run_frame(i, cam, seed, iterations)`` renders frame i, calls the filter and
    returns ((frame, rgb, length), inputs, AOV params); it is called for every frame once per iteration count 1..8. Each
    frame is checked against the reference carried over the same frames, with `mutation` applied to it."""
    out = [[run_frame(i, cam, seed + i, k) for i, cam in enumerate(cams)] for k in range(1, ITERATIONS + 1)]
    ref_hist = hist32 = None
    for i, cam in enumerate(cams):
        (frame, rgb, length), ins, a = out[-1][i]
        passes = [o[i][0][1].astype(np.float64) / np.maximum(ins[1].astype(np.float64), 1e-3) for o in out]
        res = tref.temporal_denoise(*ins, dl.primary_rays(cam, a), cam, ref_hist, iterations=ITERATIONS, mutation=mutation)
        ref_hist = res["history"]
        # the render flags are in the AOV params (the rays); the filter calls take none
        _, _, _, hist32 = dl.oracle_denoise_temporal(*ins, cam, a, hist32, reset=i == 0, iterations=1, n_threads=8)
        totals.add(check_frame(passes, frame, rgb, length, hist32.col[..., :3].astype(np.float64), ins, res, f"{what} frame {i}"), length.size)


def one_context(ctx, w, h, flags=0, **kw):
    def run_frame(i, cam, seed, iterations):
        ins, a = render(ctx, cam, w, h, seed, flags, **kw)
        return ctx.denoise_temporal(w, h, reset=i == 0, iterations=iterations), ins, a
    return run_frame


@pytest.mark.parametrize("kind", ["still", "pan", "translate", "rotate", "dolly"])
@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("name", ["c1", "cloud", "mesh"])
def test_sequences_against_the_reference(gpu_ctx, name, lens, kind):
    gpu_ctx.upload(scene_of(name))
    totals = Totals()
    for w, h in SIZES:
        cams = [camera(kind, w, h, i, lens) for i in range(FRAMES)]
        check_sequence(cams, w, h, 30, one_context(gpu_ctx, w, h), f"{name} {kind} {w}x{h}", totals)
    totals.report(f"{name} {kind} lens={lens}")


@pytest.mark.parametrize("kind", ["translate", "rotate"])
@pytest.mark.parametrize("flag", ["bvh", "no_jitter"])
def test_flags_against_the_reference(gpu_ctx, flag, kind):
    flags = {"bvh": abi.FLAG_BVH, "no_jitter": abi.FLAG_NO_JITTER}[flag]
    gpu_ctx.upload(scene_of("c1"))
    w, h = 61, 45
    totals = Totals()
    cams = [camera(kind, w, h, i, True) for i in range(FRAMES)]
    check_sequence(cams, w, h, 50, one_context(gpu_ctx, w, h, flags), f"c1 {flag} {kind}", totals)
    totals.report(f"c1 {flag} {kind}")


def test_staged_against_the_reference(gpu_ctx, parts_ctx):
    """rt3_denoise_staged_temporal over 3 parts of 2 rows with the owner last and a moving thin-lens camera: the reference's
    inputs are a one-context render of each frame, which the stage reproduces bit for bit."""
    w, h, parts, owner = 41, 23, 3, 2
    scene, _ = scenes.rtiow_four_spheres(w, h)
    gpu_ctx.upload(scene)
    for c in parts_ctx[:parts]:
        c.upload(scene)
    cams = [camera("translate", w, h, i, True) for i in range(FRAMES)]
    with Stage(parts_ctx[owner], w, h) as stage:
        def run_frame(i, cam, seed, iterations):
            ins, a = render(gpu_ctx, cam, w, h, seed)
            tag = 1000 * iterations + i
            stage_frame(parts_ctx, cam, w, h, parts, 2, stage.ptr, tag, seed)
            return parts_ctx[owner].denoise_staged_temporal(w, h, stage.ptr, tag, reset=i == 0, iterations=iterations), ins, a
        totals = Totals()
        check_sequence(cams, w, h, 70, run_frame, "staged", totals)
    totals.report("staged, 3 parts, owner last, thin lens")


# m2_towards_m1sq makes m2 - m1^2 nearly 0: the reference marks that variance ill-conditioned, which on renders holds the
# pixels it touches to the hull. It is refused on the CPU (tests/test_denoise_temporal_reference.py).
@pytest.mark.parametrize("mutation", [m for m in tref.FILTER_MUTATIONS if m != "m2_towards_m1sq"])
def test_filter_mutation_is_refused(gpu_ctx, mutation):
    """The comparison, with its exclusions, refuses the reference with one rule of steps 7-9 made wrong, on the kernels'
    output for C1 at 61x45 (a 6-frame thin-lens translation)."""
    scene, _ = scenes.rtiow_four_spheres(61, 45)
    gpu_ctx.upload(scene)
    cams = [camera("translate", 61, 45, i, True) for i in range(FRAMES)]
    with pytest.raises(AssertionError) as refused:
        check_sequence(cams, 61, 45, 90, one_context(gpu_ctx, 61, 45), "mutation", Totals(), mutation=mutation)
    print(f"{mutation}: {str(refused.value).splitlines()[0]}")
