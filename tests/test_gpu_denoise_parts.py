"""Denoising a frame rendered in parts (rt3_denoise_stage / rt3_denoise_staged): every part prepares its own rows into one
stage buffer and the owner filters the whole frame from it. The result must equal rt3_denoise of a one-context render of
the same frame bit for bit (and so the CPU restatement), over part counts, tile sizes, partial last tiles, cameras, flags,
iteration counts, sigmas, progressive renders, full-size C2 in 8 parts and parts staged from other processes; every
refusal changes nothing; the accumulators, the AOVs and the progressive state are left alone.

One context per part, all on device 0: the stage is the same device memory a peer or IPC mapping would reach, with the
same full-frame indexing (across GPUs the stores travel over NVLink)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import denoise_lib as dl
import fullsize as fs
from rt3_b200 import abi, scenes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 40, 24
MAX_PARTS = 8


@pytest.fixture(scope="module")
def parts_ctx(built):
    ctxs = [abi.Context(0) for _ in range(MAX_PARTS)]
    for c in ctxs[1:]:
        c.frame_attach(ctxs[0])
    yield ctxs
    for c in ctxs:
        c.close()


def thin_lens(cam):
    cam.lens_radius = 0.08
    cam.lens_u[:] = [1, 0, 0]
    cam.lens_v[:] = [0, 1, 0]
    return cam


def pt(w, h, spp, seed=3, depth=5, flags=0, **kw):
    return abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=depth, seed=seed, flags=flags, **kw)


def render_part(ctx, cam, w, h, spp, aov_spp, flags=0, progressive=False, seed=3, depth=5, **part):
    """The render (one shot, or two accumulating passes) and the AOVs of one part."""
    if progressive:
        half = spp // 2
        ctx.render(cam, pt(w, h, half, seed, depth, flags, **part))
        ctx.render(cam, pt(w, h, spp - half, seed, depth, flags | abi.FLAG_ACCUMULATE, first_sample=half, **part))
    else:
        ctx.render(cam, pt(w, h, spp, seed, depth, flags, **part))
    ctx.render_path_aovs(cam, pt(w, h, aov_spp, seed, depth, flags, **part))


def whole(ctx, scene, cam, w, h, spp, aov_spp, flags=0, oracle=True, seed=3, depth=5, **dn):
    """rt3_denoise of a one-context render of the frame, checked against the restatement: (frame, rgb)."""
    ctx.upload(scene)
    ctx.render(cam, pt(w, h, spp, seed, depth, flags))
    aov = ctx.render_path_aovs(cam, pt(w, h, aov_spp, seed, depth, flags))
    gpu = ctx.denoise(w, h, **dn)
    if oracle:
        cpu = dl.oracle_denoise(ctx.read_radiance(w, h), aov["albedo"], aov["normal"], aov["hit_t"], flags=flags, **dn)
        assert_same(gpu, cpu, "one-context denoise against the restatement")
    return gpu


def stage_parts(ctxs, scene, cam, w, h, parts, tile_rows, stage, tag, flags_of=lambda i: 0, upload=True, which=None, **render):
    """Renders and stages parts `which` (default all) of `parts`, part i on ctxs[i]; checks each stage's statistics."""
    for i in (range(parts) if which is None else which):
        c = ctxs[i]
        if upload:
            c.upload(scene)
        part = dict(tile_rows=tile_rows, part_index=i, part_count=parts)
        render_part(c, cam, w, h, flags=flags_of(i), **render, **part)
        c.denoise_stage(w, h, stage, tag)
        st = c.stats()
        rows = c.lib.rt3_partition_rows(h, tile_rows, i, parts)
        assert st.rows_rendered == rows and st.kernel_launches == (1 if rows else 0) and st.rays == 0


def assert_same(a, b, what):
    bad_f = int((a[0] != b[0]).sum())
    bad_rgb = int((a[1].view(np.uint32) != b[1].view(np.uint32)).sum())
    assert bad_f == 0 and bad_rgb == 0, f"{what}: {bad_f} pixels and {bad_rgb} floats differ"


class Stage:
    """A stage on the owner's device, freed on exit."""

    def __init__(self, owner, w, h):
        self.owner, self.words = owner, abi.denoise_stage_words(w, h)
        self.ptr = owner.frame_alloc(self.words)

    def read(self):
        return self.owner.buffer_read(self.ptr, np.zeros(self.words, np.uint32))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.owner.frame_free(self.ptr)


SPLITS = [(1, 8, 40, 24), (2, 1, 40, 24), (3, 2, 41, 23), (3, 8, 37, 21)]   # (parts, tile_rows, w, h): 23 and 21 leave a partial last tile
FLAGS = {"none": lambda i: 0, "no_gamma": lambda i: abi.FLAG_NO_GAMMA, "bvh_on_odd_parts": lambda i: abi.FLAG_BVH if i % 2 else 0}


@pytest.mark.parametrize("flag", list(FLAGS))
@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("parts,tile_rows,w,h", SPLITS)
def test_staged_equals_one_context_denoise(gpu_ctx, parts_ctx, parts, tile_rows, w, h, lens, flag):
    scene, cam = scenes.rtiow_four_spheres(w, h)
    if lens:
        cam = thin_lens(cam)
    with Stage(parts_ctx[0], w, h) as stage:
        stage_parts(parts_ctx, scene, cam, w, h, parts, tile_rows, stage.ptr, 11, FLAGS[flag], spp=6, aov_spp=3)
        for iterations in (1, 8):
            ref = whole(gpu_ctx, scene, cam, w, h, 6, 3, FLAGS[flag](0), iterations=iterations)
            got = parts_ctx[0].denoise_staged(w, h, stage.ptr, 11, iterations=iterations)
            assert_same(got, ref, f"{parts} parts of {tile_rows} rows, iterations {iterations}")
            st = parts_ctx[0].stats()
            assert st.kernel_launches == 1 + iterations and st.rays == 0 and st.device_ms > 0


@pytest.mark.parametrize("dn", [dict(sigma_luminance=0.5, sigma_normal=7.0, sigma_depth=0.05), dict(iterations=8, sigma_luminance=40.0, sigma_normal=1.0, sigma_depth=10.0)])
def test_non_default_parameters(gpu_ctx, parts_ctx, dn):
    w, h = 61, 45
    scene, cam = scenes.rtiow_four_spheres(w, h)
    ref = whole(gpu_ctx, scene, cam, w, h, 4, 2, **dn)
    with Stage(parts_ctx[0], w, h) as stage:
        stage_parts(parts_ctx, scene, cam, w, h, 3, 4, stage.ptr, 5, spp=4, aov_spp=2)
        assert_same(parts_ctx[0].denoise_staged(w, h, stage.ptr, 5, **dn), ref, str(dn))


def test_progressive_render_in_parts_equals_one_shot(gpu_ctx, parts_ctx):
    """Two accumulating passes per part denoise exactly like one pass of all the samples on one context."""
    scene, cam = scenes.rtiow_four_spheres(W, H)
    ref = whole(gpu_ctx, scene, cam, W, H, 8, 3)
    with Stage(parts_ctx[0], W, H) as stage:
        stage_parts(parts_ctx, scene, cam, W, H, 3, 2, stage.ptr, 9, spp=8, aov_spp=3, progressive=True)
        assert_same(parts_ctx[0].denoise_staged(W, H, stage.ptr, 9), ref, "progressive in parts")


def test_c2_full_size_in_eight_parts(gpu_ctx, parts_ctx):
    c = fs.CONFIGS["c2"]
    w, h = c["w"], c["h"]
    scene, cam = c["scene"](w, h)
    ref = whole(gpu_ctx, scene, cam, w, h, 2, 2, c["flags"], oracle=False, seed=1, depth=c["depth"])
    with Stage(parts_ctx[0], w, h) as stage:
        stage_parts(parts_ctx, scene, cam, w, h, 8, 1, stage.ptr, 2, lambda i: c["flags"], spp=2, aov_spp=2, seed=1, depth=c["depth"])
        assert_same(parts_ctx[0].denoise_staged(w, h, stage.ptr, 2), ref, "C2 in 8 parts")


CHILD = r"""
import sys
sys.path.insert(0, {root!r})
import rt3_b200
from rt3_b200 import abi, scenes
handle = bytes.fromhex(sys.argv[1])
part, parts = int(sys.argv[2]), int(sys.argv[3])
scene, cam = scenes.rtiow_cover({w}, {h})
ctx = abi.Context(0)
ctx.upload(scene)
stage = ctx.frame_import(handle)
kw = dict(mode=abi.MODE_PATHTRACE, max_depth=6, seed=4, tile_rows={tile}, part_index=part, part_count=parts)
ctx.render(cam, abi.make_params({w}, {h}, spp=4, **kw))
ctx.render_path_aovs(cam, abi.make_params({w}, {h}, spp=2, **kw))
ctx.denoise_stage({w}, {h}, stage, {tag})
ctx.stats()  # waits for the stage's stores
ctx.frame_release(stage)
ctx.close()
"""


def test_parts_staged_by_other_processes(gpu_ctx, parts_ctx):
    """The owner stages part 0; two child processes map the stage over CUDA IPC and stage parts 1 and 2."""
    w, h, tile, tag = 96, 64, 2, 123456789012345
    scene, cam = scenes.rtiow_cover(w, h)
    ref = whole(gpu_ctx, scene, cam, w, h, 4, 2, oracle=False, seed=4, depth=6)
    owner = parts_ctx[0]
    with Stage(owner, w, h) as stage:
        handle = owner.frame_export(stage.ptr)
        stage_parts(parts_ctx, scene, cam, w, h, 3, tile, stage.ptr, tag, spp=4, aov_spp=2, seed=4, depth=6, which=[0])
        code = CHILD.format(root=ROOT, w=w, h=h, tile=tile, tag=tag)
        for part in (1, 2):
            out = subprocess.run([sys.executable, "-c", code, handle.hex(), str(part), "3"], capture_output=True, text=True, timeout=300)
            assert out.returncode == 0, out.stderr[-2000:]
        assert_same(owner.denoise_staged(w, h, stage.ptr, tag), ref, "parts from three processes")


def raw_staged(ctx, w, h, stage_ptr, tag, **dn):
    """rt3_denoise_staged into sentinel-filled host arrays: (status, frame, rgb)."""
    frame = np.full((h, w), 0xDEADBEEF, np.uint32)
    rgb = np.full((h, w, 3), -7.0, np.float32)
    p = abi.denoise_params(w, h, **dn)
    rc = ctx.lib.rt3_denoise_staged(ctx.handle, C.byref(p), tag, C.c_void_p(stage_ptr), frame.ctypes.data, rgb.ctypes.data)
    return rc, frame, rgb


def test_stage_refusals_change_nothing(built):
    ctx = abi.Context(0)
    try:
        scene, cam = scenes.rtiow_four_spheres(W, H)
        ctx.upload(scene)
        with Stage(ctx, W, H) as stage:
            refused = []

            def refuse(match, ptr=stage.ptr, w=W, **dn):
                before = stage.read()
                with pytest.raises(abi.Rt3Error, match=match):
                    ctx.denoise_stage(w, H, ptr, 1, **dn)
                assert np.array_equal(stage.read(), before), f"{match}: the refused call wrote to the stage"
                refused.append(match)

            part = dict(tile_rows=2, part_index=1, part_count=2)
            refuse("needs a path-traced render")                       # nothing rendered yet
            ctx.render(cam, pt(W, H, 4, **part))
            refuse("rt3_render_path_aovs")                             # no AOVs
            ctx.render_path_aovs(cam, pt(W, H, 2, **part))
            ctx.denoise_stage(W, H, stage.ptr, 1)                      # the good call
            ctx.stats()
            stage_rows = stage.read()
            for bad in (dict(iterations=0), dict(sigma_luminance=0.0), dict(sigma_normal=2.5)):
                refuse("rt3_denoise_stage: ", **bad)
            refuse("frame was", w=W + 1)
            refuse("device_stage is NULL", ptr=0)
            ctx.render_path_aovs(cam, pt(W, H, 2, tile_rows=2, part_index=0, part_count=2))
            refuse("partition")                                        # AOVs of another part
            ctx.render_path_aovs(cam, pt(W, H, 2, tile_rows=4, part_index=1, part_count=2))
            refuse("partition")                                        # ... of other tiles
            ctx.render_path_aovs(cam, pt(W, H, 2))
            refuse("partition")                                        # ... of the whole frame
            ctx.render_path_aovs(cam, pt(W + 2, H, 2, **part))
            refuse("AOVs are")                                         # ... of another size
            ctx.render_path_aovs(abi.reference_camera(W, H, focal_length=1.5), pt(W, H, 2, **part))
            refuse("different cameras")                                # ... of another camera
            ctx.render_path_aovs(cam, pt(W, H, 2, **part))
            ctx.render(abi.reference_camera(W, H, focal_length=1.5), pt(W, H, 4, flags=abi.FLAG_ACCUMULATE, first_sample=4, **part))
            refuse("different cameras")                                # accumulated passes of two cameras
            ctx.render(cam, pt(W, H, 4, **part))
            ctx.upload(scene)
            ctx.render(cam, pt(W, H, 4, **part))
            refuse("another scene upload")                             # AOVs of the previous upload
            ctx.render_path_aovs(cam, pt(W, H, 2, **part))
            assert len(refused) == 14
            # the state the refusals saw is the one they left: the same render and AOVs stage the same bits
            ctx.denoise_stage(W, H, stage.ptr, 1)
            ctx.stats()
            assert np.array_equal(stage.read(), stage_rows)
    finally:
        ctx.close()


def test_staged_refusals_change_nothing(gpu_ctx, parts_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    ref = whole(gpu_ctx, scene, cam, W, H, 4, 2, oracle=False)
    owner, parts, tile = parts_ctx[0], 3, 2
    kw = dict(spp=4, aov_spp=2)
    with Stage(owner, W, H) as stage:
        def refuse(match, tag=1, ctx=owner):
            rc, frame, rgb = raw_staged(ctx, W, H, stage.ptr, tag)
            msg = ctx.lib.rt3_last_error().decode()
            assert rc == -1, msg                                          # RT3_ERR_INVALID
            assert match in msg, msg
            assert (frame == 0xDEADBEEF).all() and (rgb == -7.0).all(), f"{match}: the refused call wrote its outputs"

        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 1, which=[0, 1], **kw)
        fresh = abi.Context(0)
        try:
            refuse("rt3_denoise_staged needs a path-traced render", ctx=fresh)   # an owner without a render
        finally:
            fresh.close()
        refuse("row 4 (and 8 rows in all, of 24)")                   # part 2 (rows 4, 5, 10, 11, ...) never staged
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 1, which=[2], **kw)
        assert_same(owner.denoise_staged(W, H, stage.ptr, 1), ref, "after the missing part")
        refuse("row 0 (and 24 rows in all, of 24)", tag=2)           # every row is of frame 1
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 2, upload=False, which=[1, 2], **kw)
        refuse("row 0 (and 8 rows in all", tag=2)                    # part 0's rows are stale
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 2, upload=False, which=[0], **kw)
        assert_same(owner.denoise_staged(W, H, stage.ptr, 2), ref, "after the stale part")
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 2, upload=False, which=[1], seed=4, **kw)
        refuse("row 2 (and 8 rows in all", tag=2)                    # part 1 rendered with another seed
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 2, upload=False, which=[1], spp=5, aov_spp=2)
        refuse("row 2 (and 8 rows in all", tag=2)                    # ... with another spp
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 2, upload=False, which=[1], spp=4, aov_spp=3)
        refuse("row 2 (and 8 rows in all", tag=2)                    # ... AOVs of another spp
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 2, upload=False, which=[1], **kw)
        assert_same(owner.denoise_staged(W, H, stage.ptr, 2), ref, "after the part with other parameters")


def test_state_is_left_alone(gpu_ctx, parts_ctx):
    """Neither call touches the accumulators, the AOVs or the progressive state of a part."""
    scene, cam = scenes.rtiow_four_spheres(W, H)
    parts, tile, k = 3, 2, 4
    owner = parts_ctx[0]
    with Stage(owner, W, H) as stage:
        stage_parts(parts_ctx, scene, cam, W, H, parts, tile, stage.ptr, 3, spp=k, aov_spp=2)
        radiance = [c.read_radiance(W, H) for c in parts_ctx[:parts]]
        first = owner.denoise_staged(W, H, stage.ptr, 3)
        for i, c in enumerate(parts_ctx[:parts]):
            assert np.array_equal(c.read_radiance(W, H).view(np.uint32), radiance[i].view(np.uint32)), f"part {i}: radiance changed"
            c.denoise_stage(W, H, stage.ptr, 3)                     # the same render and AOVs stage the same rows again
            c.stats()
        assert_same(owner.denoise_staged(W, H, stage.ptr, 3), first, "staged twice")
        # an accumulating pass continues the render as if neither call had happened
        for i, c in enumerate(parts_ctx[:parts]):
            c.render(cam, pt(W, H, k, flags=abi.FLAG_ACCUMULATE, first_sample=k, tile_rows=tile, part_index=i, part_count=parts))
            c.denoise_stage(W, H, stage.ptr, 4)
            c.stats()
        ref = whole(gpu_ctx, scene, cam, W, H, 2 * k, 2, oracle=False)
        assert_same(owner.denoise_staged(W, H, stage.ptr, 4), ref, "after an accumulating pass")
    # a one-context render staged as a single part: rt3_denoise before and after agree, and equal the staged frame
    gpu_ctx.upload(scene)
    gpu_ctx.render(cam, pt(W, H, k))
    gpu_ctx.render_path_aovs(cam, pt(W, H, 2))
    before = gpu_ctx.denoise(W, H)
    with Stage(gpu_ctx, W, H) as stage:
        gpu_ctx.denoise_stage(W, H, stage.ptr, 8)
        gpu_ctx.stats()
        assert_same(gpu_ctx.denoise_staged(W, H, stage.ptr, 8), before, "single part")
    assert_same(gpu_ctx.denoise(W, H), before, "rt3_denoise after the staged calls")
