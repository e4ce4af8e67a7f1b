"""Temporal accumulation for a frame rendered in parts (rt3_denoise_stage on every part, rt3_denoise_staged_temporal on the
stage's owner): at every frame of camera sequences the owner's (frame, rgb, history length) must equal rt3_denoise_temporal
over one-context renders of the same frames, carried over the same sequence, bit for bit (and, through the one-context
frames, the CPU restatement). Covered: part counts, tile sizes, partial last tiles, an owner that is the first or the last
part, pinhole and thin-lens cameras, flags, non-default parameters, progressive parts, full-size C2 in 8 parts and parts
staged by other processes; the contracts (no history: rt3_denoise_staged; a still camera: n = the call count; a new upload
or size: n = 1; one history shared with rt3_denoise_temporal); every refusal without a change; the other calls' state left
alone.

One context per part, all on device 0, as in tests/test_gpu_denoise_parts.py."""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import fullsize as fs
from rt3_b200 import abi, scenes
from test_gpu_denoise_parts import FLAGS, SPLITS, Stage, render_part, whole
from test_gpu_denoise_temporal import Sequence, motion

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 40, 24
MAX_PARTS = 8
f32 = np.float32


@pytest.fixture(scope="module")
def parts_ctx(built):
    ctxs = [abi.Context(0) for _ in range(MAX_PARTS)]
    for c in ctxs[1:]:
        c.frame_attach(ctxs[0])
    yield ctxs
    for c in ctxs:
        c.close()


def assert_same(got, want, what):
    bad = [int((g.view(np.uint32) != r.view(np.uint32)).sum()) for g, r in zip(got, want)]
    assert bad == [0] * len(want), f"{what}: {bad} pixels / rgb floats / history lengths differ"


def stage_frame(ctxs, cam, w, h, parts, tile_rows, stage_ptr, tag, seed, which=None, flags_of=lambda i: 0, spp=4, aov_spp=2, depth=5, progressive=False):
    """Part i of `parts` (all, or those in `which`) renders the frame on ctxs[i] with `seed` and stages it for `tag`."""
    for i in (range(parts) if which is None else which):
        c = ctxs[i]
        render_part(c, cam, w, h, spp, aov_spp, flags=flags_of(i), progressive=progressive, seed=seed, depth=depth, tile_rows=tile_rows, part_index=i,
                    part_count=parts)
        c.denoise_stage(w, h, stage_ptr, tag)
        c.stats()  # waits for the stage's stores


def check_stats(ctx, dn):
    st = ctx.stats()
    assert st.kernel_launches == 2 + dn.get("iterations", 5) and st.rays == 0 and st.device_ms > 0


def run_sequence(one, ctxs, scene, w, h, parts, tile_rows, owner, cams, seed=10, oracle=True, flags_of=lambda i: 0, spp=4, aov_spp=2, depth=5,
                 progressive=False, **dn):
    """Frames `cams` with seeds seed, seed + 1, ...: rendered whole on `one` (rt3_denoise_temporal, checked against the
    restatement when `oracle`) and in `parts` on ctxs (rt3_denoise_staged_temporal on ctxs[owner]); returns the lengths."""
    seq = Sequence(one, w, h, spp=spp, aov_spp=aov_spp, depth=depth, flags=flags_of(0), **dn)
    one.upload(scene)
    for c in ctxs[:parts]:
        c.upload(scene)
    lengths = []
    with Stage(ctxs[owner], w, h) as stage:
        for i, cam in enumerate(cams):
            reset = i == 0
            if oracle:
                ref, cpu = seq.frame(cam, seed + i, reset)
                assert_same(ref, cpu, f"one-context frame {i} against the restatement")
            else:
                seq.render(cam, seed + i)
                ref = one.denoise_temporal(w, h, reset=reset, **dn)
            stage_frame(ctxs, cam, w, h, parts, tile_rows, stage.ptr, 100 + i, seed + i, flags_of=flags_of, spp=spp, aov_spp=aov_spp, depth=depth,
                        progressive=progressive)
            got = ctxs[owner].denoise_staged_temporal(w, h, stage.ptr, 100 + i, reset=reset, **dn)
            assert_same(got, ref, f"{parts} parts of {tile_rows} rows, owner {owner}, frame {i}")
            check_stats(ctxs[owner], dn)
            lengths.append(got[2])
    return lengths


OWNERS = {"pinhole_owner_first": (False, lambda parts: 0), "thin_lens_owner_last": (True, lambda parts: parts - 1)}


@pytest.mark.parametrize("setup", list(OWNERS))
@pytest.mark.parametrize("parts,tile_rows,w,h", SPLITS)
@pytest.mark.parametrize("kind", ["still", "pan", "translate", "rotate"])
def test_sequences_equal_one_context(gpu_ctx, parts_ctx, kind, parts, tile_rows, w, h, setup):
    lens, owner = OWNERS[setup]
    scene, _ = scenes.rtiow_four_spheres(w, h)
    lengths = run_sequence(gpu_ctx, parts_ctx, scene, w, h, parts, tile_rows, owner(parts), [motion(kind, w, h, i, lens) for i in range(4)])
    assert lengths[-1].max() > 1.0, "no pixel kept any history"


FLAG_CASES = dict(FLAGS, no_jitter=lambda i: abi.FLAG_NO_JITTER)


@pytest.mark.parametrize("flag", [k for k in FLAG_CASES if k != "none"])
@pytest.mark.parametrize("parts,tile_rows,w,h,owner", [(2, 1, 40, 24, 0), (3, 2, 41, 23, 2)])
def test_flags(gpu_ctx, parts_ctx, parts, tile_rows, w, h, owner, flag):
    scene, _ = scenes.rtiow_four_spheres(w, h)
    run_sequence(gpu_ctx, parts_ctx, scene, w, h, parts, tile_rows, owner, [motion("rotate", w, h, i, True) for i in range(4)], flags_of=FLAG_CASES[flag])


def test_non_default_parameters(gpu_ctx, parts_ctx):
    dn = dict(alpha_color=0.5, alpha_moments=0.05, depth_tolerance=0.01, normal_cos=0.99, iterations=2, sigma_luminance=0.5, sigma_normal=7.0)
    scene, _ = scenes.rtiow_four_spheres(61, 45)
    run_sequence(gpu_ctx, parts_ctx, scene, 61, 45, 3, 4, 1, [motion("translate", 61, 45, i) for i in range(5)], **dn)


def test_progressive_parts(gpu_ctx, parts_ctx):
    """Two accumulating passes per part, against one pass of all the samples on one context."""
    scene, _ = scenes.rtiow_four_spheres(W, H)
    run_sequence(gpu_ctx, parts_ctx, scene, W, H, 3, 2, 2, [motion("pan", W, H, i) for i in range(4)], spp=8, aov_spp=3, progressive=True)


def test_c2_full_size_in_eight_parts(gpu_ctx, parts_ctx):
    c = fs.CONFIGS["c2"]
    w, h = c["w"], c["h"]
    scene, cam = c["scene"](w, h)
    run_sequence(gpu_ctx, parts_ctx, scene, w, h, 8, 1, 7, [motion("translate", w, h, i, base=cam) for i in range(3)], seed=1, oracle=False,
                 flags_of=lambda i: c["flags"], spp=2, aov_spp=2, depth=c["depth"])


CHILD = r"""
import json
import sys
sys.path.insert(0, {root!r})
import rt3_b200
from rt3_b200 import abi, scenes
handle = bytes.fromhex(sys.argv[1])
part, parts = int(sys.argv[2]), int(sys.argv[3])
scene, _ = scenes.rtiow_cover({w}, {h})
ctx = abi.Context(0)
ctx.upload(scene)
stage = ctx.frame_import(handle)
for line in sys.stdin:
    job = json.loads(line)
    cam = abi.make_camera(*job["cam"])
    kw = dict(mode=abi.MODE_PATHTRACE, max_depth=6, seed=job["seed"], tile_rows={tile}, part_index=part, part_count=parts)
    ctx.render(cam, abi.make_params({w}, {h}, spp=4, **kw))
    ctx.render_path_aovs(cam, abi.make_params({w}, {h}, spp=2, **kw))
    ctx.denoise_stage({w}, {h}, stage, job["tag"])
    ctx.stats()  # waits for the stage's stores
    print("staged", flush=True)
ctx.frame_release(stage)
ctx.close()
"""


def test_parts_staged_by_other_processes(gpu_ctx, parts_ctx):
    """The owner stages part 0 of every frame; two child processes map the stage over CUDA IPC and stage parts 1 and 2."""
    w, h, tile, parts = 96, 64, 2, 3
    scene, base = scenes.rtiow_cover(w, h)
    seq = Sequence(gpu_ctx, w, h, spp=4, aov_spp=2, depth=6)
    gpu_ctx.upload(scene)
    owner = parts_ctx[0]
    owner.upload(scene)
    with Stage(owner, w, h) as stage, tempfile.TemporaryFile("w+") as err:
        code, handle = CHILD.format(root=ROOT, w=w, h=h, tile=tile), owner.frame_export(stage.ptr).hex()
        children = [subprocess.Popen([sys.executable, "-c", code, handle, str(part), str(parts)], stdin=subprocess.PIPE,
                                     stdout=subprocess.PIPE, stderr=err, text=True) for part in (1, 2)]
        try:
            for i in range(3):
                cam = motion("translate", w, h, i, base=base)
                seed, tag = 4 + i, 123456789012345 + i
                seq.render(cam, seed)
                ref = gpu_ctx.denoise_temporal(w, h, reset=i == 0)
                job = {"cam": [list(cam.origin), list(cam.horizontal), list(cam.vertical), list(cam.lower_left_corner)], "seed": seed, "tag": tag}
                for child in children:
                    child.stdin.write(json.dumps(job) + "\n")
                    child.stdin.flush()
                stage_frame(parts_ctx, cam, w, h, parts, tile, stage.ptr, tag, seed, which=[0], depth=6)
                for child in children:
                    line = None
                    while line not in ("staged\n", ""):                 # "": the child ended
                        line = child.stdout.readline()
                    err.seek(0)
                    assert line, err.read()[-2000:]
                assert_same(owner.denoise_staged_temporal(w, h, stage.ptr, tag, reset=i == 0), ref, f"parts from three processes, frame {i}")
        finally:
            for child in children:
                child.stdin.close()
            codes = [child.wait(timeout=300) for child in children]
        assert codes == [0, 0]


def test_first_call_and_reset_equal_staged_and_still_camera_counts_calls(built, parts_ctx):
    """On an owner that never had a history, and after a reset, the call is rt3_denoise_staged; under NO_JITTER a still
    camera sees the same surface point in every frame, so every pixel's history grows by one per call."""
    scene, cam = scenes.rtiow_four_spheres(W, H)
    owner = abi.Context(0)
    try:
        ctxs = [parts_ctx[1], owner, parts_ctx[2]]                  # the owner is part 1 of 3
        for c in ctxs:
            c.upload(scene)
        flags = lambda i: abi.FLAG_NO_JITTER
        with Stage(owner, W, H) as stage:
            for i in range(5):
                stage_frame(ctxs, cam, W, H, 3, 2, stage.ptr, i, 40 + i, flags_of=flags)
                plain = owner.denoise_staged(W, H, stage.ptr, i)
                got = owner.denoise_staged_temporal(W, H, stage.ptr, i, reset=i == 3)
                if i in (0, 3):
                    assert_same(got[:2], plain, f"frame {i}: no history")
                assert np.all(got[2] == (i + 1 if i < 3 else i - 2)), np.unique(got[2])
    finally:
        owner.close()


def test_new_upload_or_size_drops_the_history(built, parts_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    ctxs = parts_ctx[:2]
    flags = lambda i: abi.FLAG_NO_JITTER
    for c in ctxs:
        c.upload(scene)
    with Stage(ctxs[0], W, H) as stage:
        for i in range(2):
            stage_frame(ctxs, cam, W, H, 2, 1, stage.ptr, i, 1 + i, flags_of=flags)
            assert np.all(ctxs[0].denoise_staged_temporal(W, H, stage.ptr, i, reset=i == 0)[2] == i + 1)
        for c in ctxs:                                             # same scene, new upload on every part
            c.upload(scene)
        stage_frame(ctxs, cam, W, H, 2, 1, stage.ptr, 2, 3, flags_of=flags)
        assert np.all(ctxs[0].denoise_staged_temporal(W, H, stage.ptr, 2)[2] == 1)
        stage_frame(ctxs, cam, W, H, 2, 1, stage.ptr, 3, 4, flags_of=flags)
        assert np.all(ctxs[0].denoise_staged_temporal(W, H, stage.ptr, 3)[2] == 2)
    _, cam2 = scenes.rtiow_four_spheres(W + 3, H)
    with Stage(ctxs[0], W + 3, H) as stage:                        # another size
        stage_frame(ctxs, cam2, W + 3, H, 2, 1, stage.ptr, 4, 5, flags_of=flags)
        assert np.all(ctxs[0].denoise_staged_temporal(W + 3, H, stage.ptr, 4)[2] == 1)


def test_history_is_shared_with_one_context_frames(gpu_ctx, parts_ctx):
    """Frames 0 and 2 rendered whole on the owner (rt3_denoise_temporal), 1 and 3 in parts (rt3_denoise_staged_temporal):
    the bits of a sequence of one-context frames."""
    w, h, parts, tile = 41, 23, 3, 2
    scene, _ = scenes.rtiow_four_spheres(w, h)
    seq = Sequence(gpu_ctx, w, h)
    gpu_ctx.upload(scene)
    owner = parts_ctx[2]
    for c in parts_ctx[:parts]:
        c.upload(scene)
    mixed = Sequence(owner, w, h)
    with Stage(owner, w, h) as stage:
        for i in range(4):
            cam = motion("rotate", w, h, i, lens=True)
            ref, cpu = seq.frame(cam, 70 + i, reset=i == 0)
            assert_same(ref, cpu, f"one-context frame {i} against the restatement")
            if i % 2 == 0:
                mixed.render(cam, 70 + i)
                got = owner.denoise_temporal(w, h, reset=i == 0)
            else:
                stage_frame(parts_ctx, cam, w, h, parts, tile, stage.ptr, i, 70 + i)
                got = owner.denoise_staged_temporal(w, h, stage.ptr, i)
            assert_same(got, ref, f"mixed sequence, frame {i}")


def raw_staged_temporal(ctx, w, h, stage_ptr, tag, null_params=False, **kw):
    """rt3_denoise_staged_temporal into sentinel-filled host arrays: (status, message, frame, rgb, length)."""
    frame = np.full((h, w), 0xDEADBEEF, np.uint32)
    rgb = np.full((h, w, 3), -7.0, f32)
    length = np.full((h, w), -7.0, f32)
    p = abi.denoise_temporal_params(w, h, **kw)
    rc = ctx.lib.rt3_denoise_staged_temporal(ctx.handle, None if null_params else C.byref(p), tag, C.c_void_p(stage_ptr), frame.ctypes.data,
                                             rgb.ctypes.data, length.ctypes.data)
    return rc, ctx.lib.rt3_last_error().decode(), frame, rgb, length


def test_refusals_change_nothing(built, parts_ctx):
    """Frame A, every refusal, frame B: B's bits equal those of A then B without the refusals, and no refusal wrote its
    outputs or the stage."""
    scene, _ = scenes.rtiow_four_spheres(W, H)
    parts, tile = 3, 2
    owner = parts_ctx[parts - 1]
    cam_a, cam_b = motion("translate", W, H, 0), motion("translate", W, H, 1)
    for c in parts_ctx[:parts]:
        c.upload(scene)
    refused = []

    def refuse(match, ctx=owner, ptr=None, tag=2, w=W, **kw):
        before = stage.read()
        rc, msg, frame, rgb, length = raw_staged_temporal(ctx, w, H, stage.ptr if ptr is None else ptr, tag, **kw)
        assert rc == -1, msg                                       # RT3_ERR_INVALID
        assert f"rt3_denoise_staged_temporal{match}" in msg, msg
        assert (frame == 0xDEADBEEF).all() and (rgb == -7.0).all() and (length == -7.0).all(), f"{match}: the refused call wrote its outputs"
        assert np.array_equal(stage.read(), before), f"{match}: the refused call wrote to the stage"
        refused.append(match)

    with Stage(owner, W, H) as stage:
        fresh = abi.Context(0)
        try:
            fresh.upload(scene)
            refuse(" needs a path-traced render", ctx=fresh)
            fresh.render(cam_a, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=4, max_depth=5, seed=3))
            refuse(" needs an rt3_render_path_aovs", ctx=fresh)
        finally:
            fresh.close()
        stage_frame(parts_ctx, cam_a, W, H, parts, tile, stage.ptr, 1, 20)
        a = owner.denoise_staged_temporal(W, H, stage.ptr, 1, reset=True)
        stage_frame(parts_ctx, cam_b, W, H, parts, tile, stage.ptr, 2, 21, which=[1, 2])
        refuse(": row 0 (and 8 rows in all, of 24) was not staged")   # part 0 (rows 0, 1, 6, 7, ...) is still of frame A
        stage_frame(parts_ctx, cam_b, W, H, parts, tile, stage.ptr, 2, 21, which=[0])
        refuse(": row 0 (and 24 rows in all, of 24)", tag=3)         # every row is stale for tag 3
        refuse(": params is NULL", null_params=True)
        refuse(": device_stage is NULL", ptr=0)
        refuse(": the last path-traced frame was", w=W + 1)
        for bad, msg in ((dict(iterations=0), "iterations"), (dict(sigma_normal=2.5), "sigma_normal"), (dict(alpha_color=0.0), "alpha_color"),
                         (dict(alpha_moments=float("nan")), "alpha_moments"), (dict(depth_tolerance=float("inf")), "depth_tolerance"),
                         (dict(normal_cos=1.01), "normal_cos")):
            refuse(f": {msg}", **bad)
        stage_frame(parts_ctx, cam_b, W, H, parts, tile, stage.ptr, 2, 22, which=[1])
        refuse(": row 2 (and 8 rows in all, of 24)")                 # part 1 rendered with another seed
        stage_frame(parts_ctx, cam_b, W, H, parts, tile, stage.ptr, 2, 21, which=[1])
        assert len(refused) == 14
        b = owner.denoise_staged_temporal(W, H, stage.ptr, 2)
        # the same two frames without the refusals in between
        stage_frame(parts_ctx, cam_a, W, H, parts, tile, stage.ptr, 1, 20)
        assert_same(owner.denoise_staged_temporal(W, H, stage.ptr, 1, reset=True), a, "frame A again")
        stage_frame(parts_ctx, cam_b, W, H, parts, tile, stage.ptr, 2, 21)
        assert_same(owner.denoise_staged_temporal(W, H, stage.ptr, 2), b, "frame B after the refusals")
        assert b[2].max() > 1.0


def test_other_state_is_left_alone(gpu_ctx, parts_ctx):
    """The parts' radiance and AOVs, rt3_denoise_staged, a following RT3_FLAG_ACCUMULATE pass and rt3_denoise behave as
    if the temporal calls had not happened."""
    scene, cam = scenes.rtiow_four_spheres(W, H)
    parts, tile, k = 3, 2, 4
    owner = parts_ctx[0]
    for c in parts_ctx[:parts]:
        c.upload(scene)
    with Stage(owner, W, H) as stage:
        stage_frame(parts_ctx, cam, W, H, parts, tile, stage.ptr, 3, 5, spp=k)
        staged = stage.read()
        radiance = [c.read_radiance(W, H) for c in parts_ctx[:parts]]
        plain = owner.denoise_staged(W, H, stage.ptr, 3)
        for reset in (True, False, False):
            owner.denoise_staged_temporal(W, H, stage.ptr, 3, reset=reset)
        assert np.array_equal(stage.read(), staged), "the calls wrote to the stage"
        assert_same(owner.denoise_staged(W, H, stage.ptr, 3), plain, "rt3_denoise_staged after the temporal calls")
        for i, c in enumerate(parts_ctx[:parts]):
            assert np.array_equal(c.read_radiance(W, H).view(np.uint32), radiance[i].view(np.uint32)), f"part {i}: radiance changed"
            c.denoise_stage(W, H, stage.ptr, 3)                    # the same render and AOVs stage the same bits again
            c.stats()
        assert np.array_equal(stage.read(), staged), "the render or the AOVs changed"
        for i, c in enumerate(parts_ctx[:parts]):
            c.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=k, max_depth=5, seed=5, flags=abi.FLAG_ACCUMULATE, first_sample=k,
                                          tile_rows=tile, part_index=i, part_count=parts))
            c.denoise_stage(W, H, stage.ptr, 4)
            c.stats()
        ref = whole(gpu_ctx, scene, cam, W, H, 2 * k, 2, oracle=False, seed=5)
        assert_same(owner.denoise_staged(W, H, stage.ptr, 4), ref, "after an accumulating pass")
    # a one-context render staged as a single part: rt3_denoise before and after the temporal calls agree
    gpu_ctx.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=k, max_depth=5, seed=6))
    gpu_ctx.render_path_aovs(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=2, max_depth=5, seed=6))
    before = gpu_ctx.denoise(W, H)
    with Stage(gpu_ctx, W, H) as stage:
        gpu_ctx.denoise_stage(W, H, stage.ptr, 8)
        gpu_ctx.stats()
        first = gpu_ctx.denoise_staged_temporal(W, H, stage.ptr, 8, reset=True)
        check_stats(gpu_ctx, {})
        assert_same(first[:2], before, "single part, no history")
        gpu_ctx.denoise_staged_temporal(W, H, stage.ptr, 8, iterations=3)
        check_stats(gpu_ctx, dict(iterations=3))
    assert_same(gpu_ctx.denoise(W, H), before, "rt3_denoise after the temporal calls")
