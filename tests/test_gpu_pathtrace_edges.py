"""The path tracer at the edges of its sweep, against the CPU restatement (oracle/rt3_oracle.c) and against itself, bit for bit:
the count ladder across the padding, word, chunk, constant-bank and tile edges (sphere-only, mixed with the face/sphere id
boundary on those edges, mixed with random materials) through the sweep and the hierarchy; buried padding that moves C1 and
C2 across the bank and tile edges at their real shapes; ties across every edge and a crowd of coincident spheres that
overflows the BEAM candidate list; every hierarchy sort around its face and spp thresholds; the scheduler's edges; and a
partition that owns no rows. The scenes and the plan rules come from tests/pathtrace_edges.py; the CPU half
(tests/test_pathtrace_edges_cpu.py) checks that each scene has the property relied on here and that the cases reach all
eleven pathtrace_kernel instantiations."""
import numpy as np
import pytest

import oraclelib as ol
import pathtrace_edges as pe
from rt3_b200 import abi, scenes

pytestmark = pytest.mark.gpu


def set_env(monkeypatch, env):
    for k in ("RT3_BEAM", "RT3_BINNING", "RT3_BEAM_BVH"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def render_mode(ctx, monkeypatch, cam, params, mode):
    """Renders with one of pathtrace_edges' modes: (frame, stats)."""
    name, bvh, env = mode
    set_env(monkeypatch, env)
    p = abi.Params.from_buffer_copy(params)
    if bvh:
        p.flags |= abi.FLAG_BVH
    frame = ctx.render(cam, p)
    st = ctx.stats()
    set_env(monkeypatch, {})
    assert st.accel == int(bvh) and st.accel_stack_overflows == 0, name
    return frame, st


def assert_frame(got, want, what):
    assert np.array_equal(got, want), f"{what}: {int((got != want).sum())} pixels differ"


LADDER_CASES = [(n, form, False) for n in pe.LADDER for form in pe.FORMS] + [(769, "spheres", True), (1025, "mixed", True)]


@pytest.mark.parametrize("n,form,lens", LADDER_CASES, ids=[f"{form}-{n}" + ("-lens" if lens else "") for n, form, lens in LADDER_CASES])
def test_ladder_against_the_oracle(gpu_ctx, monkeypatch, n, form, lens):
    w, h = pe.LADDER_W, pe.LADDER_H
    scene, cam = pe.ladder_scene(n, form, w, h)
    if lens:
        cam = pe.thin_lens(cam)
    params = pe.pt(w, h, pe.LADDER_SPP, pe.LADDER_DEPTH, seed=n)
    cpu, _, rays = ol.oracle_pathtrace(scene, cam, params)
    gpu_ctx.upload(scene)
    nf, ns = pe.ladder_split(n, form)
    for mode in pe.ladder_modes(n, form):
        kernel = pe.kernel_for(nf, ns, pe.LADDER_SPP, mode[1], mode[2])
        what = f"{form} {n} ({nf} faces) {mode[0]}, pathtrace_kernel<{','.join(map(str, kernel))}>"
        frame, st = render_mode(gpu_ctx, monkeypatch, cam, params, mode)
        assert st.rays == rays, f"{what}: rays {st.rays} vs oracle {rays}"
        assert_frame(frame, cpu, what)
        if not kernel[4]:
            assert st.beam_rays == 0, what
        if not kernel[2] and not kernel[4]:   # the plain sweep tests every primitive on every ray
            assert st.sphere_tests == st.rays * ns and st.face_tests == st.rays * nf, what


@pytest.mark.parametrize("totals", [(768, 769), (1024, 1025)], ids=["bank", "tile"])
def test_buried_padding_at_c1_full_size(gpu_ctx, totals):
    """C1 at 400x225, 64 spp, depth 50: padded with buried spheres (and with buried triangles ahead of them) across an edge,
    the frame and the ray count are the unpadded render's."""
    w, h = 400, 225
    scene, cam = pe.c1_padded(4, w, h)
    params = pe.pt(w, h, 64, 50, seed=1)
    gpu_ctx.upload(scene)
    ref = gpu_ctx.render(cam, params)
    rays = gpu_ctx.stats().rays
    for total in totals:
        for faces in (0, 40):
            padded, _ = pe.c1_padded(total, w, h, faces=faces)
            gpu_ctx.upload(padded)
            assert_frame(gpu_ctx.render(cam, params), ref, f"C1 padded to {total} ({faces} buried faces)")
            assert gpu_ctx.stats().rays == rays


def test_buried_padding_at_c2_full_size(gpu_ctx):
    """Rows of C2's 1200x800 frame at 64 spp as one-row partitions: padded to 768, 769, 1024 and 1025 primitives (off the
    BEAM kernel onto the streamed sweep), the rows and their ray counts are the unpadded scene's."""
    w, h = 1200, 800
    base, cam = pe.c2_padded(485, w, h)
    rows = (96, 400, 640, 796)
    frame = np.zeros((h, w), np.uint32)

    def render_rows(scene):
        gpu_ctx.upload(scene)
        out = {}
        for y in rows:
            gpu_ctx.render(cam, pe.pt(w, h, 64, 50, seed=1, tile_rows=1, part_index=y, part_count=h), out=frame)
            out[y] = (frame[y].copy(), gpu_ctx.stats().rays)
        return out

    ref = render_rows(base)
    for total in (768, 769, 1024, 1025):
        got = render_rows(pe.c2_padded(total, w, h)[0])
        for y in rows:
            assert_frame(got[y][0], ref[y][0], f"C2 padded to {total}, row {y}")
            assert got[y][1] == ref[y][1], (total, y)


TIE_W, TIE_H, TIE_SPP, TIE_DEPTH = 48, 27, 8, 50


@pytest.fixture(scope="module")
def c1_oracle():
    scene, cam = pe.c1_padded(4, TIE_W, TIE_H)
    frame, _, rays = ol.oracle_pathtrace(scene, cam, pe.pt(TIE_W, TIE_H, TIE_SPP, TIE_DEPTH))
    return frame, rays


@pytest.mark.parametrize("name", list(pe.TIE_CASES))
def test_ties_across_every_edge(gpu_ctx, monkeypatch, c1_oracle, name):
    """The metal copies lose to the lower id everywhere: the frame is the one without them and the oracle's C1 frame."""
    (scene, cam), without = pe.tie_scene(name, TIE_W, TIE_H)
    params = pe.pt(TIE_W, TIE_H, TIE_SPP, TIE_DEPTH)
    for mode in pe.TIE_MODES:
        gpu_ctx.upload(without)
        plain, _ = render_mode(gpu_ctx, monkeypatch, cam, params, mode)
        gpu_ctx.upload(scene)
        frame, st = render_mode(gpu_ctx, monkeypatch, cam, params, mode)
        assert_frame(frame, plain, f"{name} {mode[0]}: with the copies against without")
        assert_frame(frame, c1_oracle[0], f"{name} {mode[0]}: against the oracle")
        assert st.rays == c1_oracle[1]


@pytest.fixture(scope="module")
def meshes(gpu_ctx):
    """A tessellated sphere of 1 024 faces (32 meridians, 18 parallels) and the same without its last face, each with a
    ground sphere and a glass sphere."""
    mesh = gpu_ctx.tessellate_spheres([((0.0, 0.0, -3.0), 1.0, 32, 18, (0.8, 0.3, 0.3), 0)])
    assert mesh.n_faces == 1024
    mats = np.zeros(2, abi.MATERIAL_DTYPE)
    mats["kind"] = [abi.MAT_LAMBERTIAN, abi.MAT_DIELECTRIC]
    mats["albedo"] = [(0.8, 0.8, 0.0), (1, 1, 1)]
    mats["ior"] = [1, 1.5]
    out = {}
    for nf in pe.BIN_FACES:
        out[nf] = abi.SceneArrays(faces=mesh.faces[:nf], vertices=mesh.vertices, face_entity=mesh.face_entity[:nf],
                                  face_material=np.zeros(nf, np.uint32), spheres=np.array([(0, -101, -3, 100), (1.7, 0, -2.6, 0.5)], np.float32),
                                  sphere_material=np.array([0, 1], np.uint32), materials=mats)
    return out


@pytest.mark.parametrize("spp", pe.BIN_SPP)
@pytest.mark.parametrize("nf", pe.BIN_FACES)
def test_every_hierarchy_sort(gpu_ctx, monkeypatch, meshes, nf, spp):
    """RT3_BINNING 0..3, with and without RT3_BEAM_BVH=1, around the 1 024-face and 8-spp thresholds: all frames are the oracle's.
    With 1 024 faces, RT3_BINNING=2 is the two-class per-warp sort, pathtrace_kernel<1,0,1,2,0>."""
    w, h = 40, 24
    scene, cam = meshes[nf], abi.reference_camera(w, h, focal_length=1.0)
    params = pe.pt(w, h, spp, 8, seed=spp)
    cpu, _, rays = ol.oracle_pathtrace(scene, cam, params)
    gpu_ctx.upload(scene)
    for mode in [pe.SWEEP, pe.BVH] + pe.BIN_MODES:
        kernel = pe.kernel_for(nf, 2, spp, mode[1], mode[2])
        frame, st = render_mode(gpu_ctx, monkeypatch, cam, params, mode)
        what = f"{nf} faces, {spp} spp, {mode[0]}: pathtrace_kernel<{','.join(map(str, kernel))}>"
        assert_frame(frame, cpu, what)
        assert st.rays == rays, what
        if not kernel[4]:
            assert st.beam_rays == 0, what


SCHEDULES = [(2, 2, 4, 0, 1), (3, 2, 4, 0, 1), (2, 3, 4, 0, 1),                                  # tiny frames
             (31, 2, 1, 0, 2), (8, 4, 1, 0, 1), (11, 3, 1, 0, 1), (17, 5, 3, 0, 1), (16, 16, 1, 0, 1), (257, 2, 1, 0, 2),   # 31, 32, 33, 255, 256, 257 items
             (5, 3, 4, 2 ** 31 - 1 - 4, 1),                                                # the last sample window below 2^31
             (2, 2, 65535, 0, 1)]                                                           # the largest spp of a 16-bit count


@pytest.mark.parametrize("w,h,spp,first,parts", SCHEDULES, ids=[f"{w}x{h}x{spp}@{first}/{parts}" for w, h, spp, first, parts in SCHEDULES])
def test_scheduling_edges(gpu_ctx, monkeypatch, w, h, spp, first, parts):
    """Frames of a few pixels and path-item counts around the warp (32) and the item claim (RT3_ITEM_CHUNK, 256); odd counts
    are one row of a two-row frame (the restatement takes frames of 2x2 and up), rendered as a one-row partition."""
    scene, cam = scenes.rtiow_four_spheres(w, h)
    params = pe.pt(w, h, spp, 4 if spp > 1000 else 8, seed=7, first_sample=first, tile_rows=1, part_count=parts)
    cpu, _, rays = ol.oracle_pathtrace(scene, cam, params)
    rows = slice(0, h, parts)
    gpu_ctx.upload(scene)
    for mode in (pe.SWEEP, pe.NO_BEAM, pe.BVH):
        frame, st = render_mode(gpu_ctx, monkeypatch, cam, params, mode)
        assert_frame(frame[rows], cpu[rows], f"{w}x{h} {spp} spp from {first} in {parts} parts, {mode[0]}")
        assert st.rays == rays and st.rows_rendered == len(range(h)[rows])


# a partition that owns no rows: 6 rows in tiles of 2 are 3 tiles, the 4th of 4 parts has none
ZW, ZH, ZTILE, ZPARTS = 40, 6, 2, 4


def zpart(i, spp=4, **kw):
    return pe.pt(ZW, ZH, spp, 5, seed=3, tile_rows=ZTILE, part_index=i, part_count=ZPARTS, **kw)


@pytest.fixture
def fresh_ctxs(built):
    ctxs = [abi.Context(0) for _ in range(ZPARTS)]
    for c in ctxs[1:]:
        c.frame_attach(ctxs[0])
    yield ctxs
    for c in ctxs:
        c.close()


def test_partition_without_rows_is_a_render(fresh_ctxs):
    """On a fresh context: the render writes nothing and renders no rows, its radiance is all zeros, it can be continued with
    RT3_FLAG_ACCUMULATE (from the sample it ended at only) and its rows (none) can be staged for the denoiser."""
    ctx = fresh_ctxs[3]
    assert ctx.lib.rt3_partition_rows(ZH, ZTILE, 3, ZPARTS) == 0
    scene, cam = scenes.rtiow_four_spheres(ZW, ZH)
    ctx.upload(scene)
    out = np.full((ZH, ZW), 0x12345678, np.uint32)
    ctx.render(cam, zpart(3), out=out)
    st = ctx.stats()
    assert (out == 0x12345678).all() and st.rows_rendered == 0 and st.rays == 0
    assert not ctx.read_radiance(ZW, ZH).any()
    with pytest.raises(abi.Rt3Error, match="first_sample"):
        ctx.render(cam, zpart(3, spp=2, first_sample=5, flags=abi.FLAG_ACCUMULATE))
    ctx.render(cam, zpart(3, spp=2, first_sample=4, flags=abi.FLAG_ACCUMULATE), out=out)
    assert (out == 0x12345678).all() and ctx.stats().rows_rendered == 0
    ctx.render_path_aovs(cam, zpart(3, spp=2))
    stage = fresh_ctxs[0].frame_alloc(abi.denoise_stage_words(ZW, ZH))
    try:
        ctx.denoise_stage(ZW, ZH, stage, 1)
        st = ctx.stats()
        assert st.rows_rendered == 0 and st.kernel_launches == 0
    finally:
        fresh_ctxs[0].frame_free(stage)


def test_partition_without_rows_replaces_the_previous_render(gpu_ctx):
    """After a full-frame render on the same context, a render of a part without rows is what the accumulators stand for: its
    radiance is zeros, not the earlier frame's rows, and ACCUMULATE continues it, not the earlier render."""
    scene, cam = scenes.rtiow_four_spheres(ZW, ZH)
    gpu_ctx.upload(scene)
    gpu_ctx.render(cam, pe.pt(ZW, ZH, 4, 5, seed=3))
    assert gpu_ctx.read_radiance(ZW, ZH).any()
    gpu_ctx.render(cam, zpart(3))
    assert not gpu_ctx.read_radiance(ZW, ZH).any()
    gpu_ctx.render(cam, zpart(3, spp=2, first_sample=4, flags=abi.FLAG_ACCUMULATE))
    with pytest.raises(abi.Rt3Error, match="partition"):
        gpu_ctx.render(cam, pe.pt(ZW, ZH, 2, 5, seed=3, first_sample=6, flags=abi.FLAG_ACCUMULATE))
    with pytest.raises(abi.Rt3Error, match="covers part 3 of 4"):
        gpu_ctx.denoise(ZW, ZH)


def test_staged_denoise_with_a_part_without_rows(gpu_ctx, fresh_ctxs):
    """Four parts of a 6-row frame, the last with no rows: the owner's rt3_denoise_staged equals one-context rt3_denoise."""
    scene, cam = scenes.rtiow_four_spheres(ZW, ZH)
    gpu_ctx.upload(scene)
    gpu_ctx.render(cam, pe.pt(ZW, ZH, 4, 5, seed=3))
    gpu_ctx.render_path_aovs(cam, pe.pt(ZW, ZH, 2, 5, seed=3))
    ref = gpu_ctx.denoise(ZW, ZH)
    stage = fresh_ctxs[0].frame_alloc(abi.denoise_stage_words(ZW, ZH))
    try:
        for i, c in enumerate(fresh_ctxs):
            c.upload(scene)
            c.render(cam, zpart(i))
            c.render_path_aovs(cam, zpart(i, spp=2))
            c.denoise_stage(ZW, ZH, stage, 9)
        got = fresh_ctxs[0].denoise_staged(ZW, ZH, stage, 9)
    finally:
        fresh_ctxs[0].frame_free(stage)
    assert_frame(got[0], ref[0], "staged frame")
    assert np.array_equal(got[1].view(np.uint32), ref[1].view(np.uint32)), "staged rgb differs"
