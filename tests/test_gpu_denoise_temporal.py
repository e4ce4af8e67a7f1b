"""rt3_denoise_temporal on the GPU: every frame of camera sequences bit for bit against the CPU restatement
(tests/denoise_temporal_oracle.c) fed the same read_radiance / render_path_aovs arrays and carrying its own history; the contracts
(no history: rt3_denoise; an unchanged camera: n = the call count; a pan: the entering columns start again; a new scene
upload or size: n = 1); every refusal without a change; the other calls' state left alone; quality against rt3_denoise;
the host backend."""
import numpy as np
import pytest

import denoise_lib as dl
import denoise_temporal_lib as dtl
import fullsize as fs
import oraclelib as ol
from rt3_b200 import abi, scenes
from test_gpu_path_aovs import W, H, scene_of

pytestmark = pytest.mark.gpu

f32 = np.float32


def cam_of(origin, hor, ver, llc, lens=False):
    cam = abi.make_camera(origin, hor, ver, llc)
    if lens:
        cam.lens_radius = 0.08
        cam.lens_u[:] = [1, 0, 0]
        cam.lens_v[:] = [0, 1, 0]
    return cam


def rot_y(a, v):
    R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    return f32(R @ np.asarray(v, np.float64))


def motion(kind, w, h, i, lens=False, step=1.0, base=None):
    """The camera of frame i of a sequence: the reference camera (or `base`), then `still`, an image-plane `pan` of `step`
    pixels per frame (llc moved by step hor / (W - 1)), a `translate` of the whole camera to the right (parallax), a
    `rotate` about the vertical axis through the camera's origin, or an `orbit` of 0.005 rad per frame about the vertical
    axis through (0, 0, -1)."""
    base = base or abi.reference_camera(w, h)
    o, hor, ver, llc = (np.array(getattr(base, k)[:], f32) for k in ("origin", "horizontal", "vertical", "lower_left_corner"))
    if kind == "pan":
        llc = llc + f32(step * i) * hor / f32(w - 1)
    elif kind == "translate":
        shift = np.array([0.03 * i, 0.0, 0.0], f32)
        o, llc = o + shift, llc + shift
    elif kind == "rotate":
        a = 0.01 * i
        hor, ver, llc = rot_y(a, hor), rot_y(a, ver), rot_y(a, llc - o) + o
    elif kind == "orbit":
        a, pivot = 0.005 * i, np.array([0, 0, -1], f32)
        hor, ver, o, llc = rot_y(a, hor), rot_y(a, ver), rot_y(a, o - pivot) + pivot, rot_y(a, llc - pivot) + pivot
    else:
        assert kind == "still", kind
    return cam_of(o, hor, ver, llc, lens)


class Sequence:
    """Renders frames on `ctx` and runs rt3_denoise_temporal and the restatement side by side, the restatement carrying
    its own history."""

    def __init__(self, ctx, w, h, spp=4, aov_spp=2, depth=5, flags=0, scene_tag=0, **dn):
        self.ctx, self.w, self.h, self.spp, self.aov_spp, self.depth, self.flags, self.dn = ctx, w, h, spp, aov_spp, depth, flags, dn
        self.history, self.scene = None, scene_tag

    def render(self, cam, seed):
        p = abi.make_params(self.w, self.h, mode=abi.MODE_PATHTRACE, spp=self.spp, max_depth=self.depth, seed=seed, flags=self.flags)
        a = abi.make_params(self.w, self.h, mode=abi.MODE_PATHTRACE, spp=self.aov_spp, max_depth=self.depth, seed=seed, flags=self.flags)
        self.ctx.render(cam, p)
        self.aov = self.ctx.render_path_aovs(cam, a)
        self.aov_params, self.cam = a, cam
        self.rgb = self.ctx.read_radiance(self.w, self.h)

    def denoise(self, reset=False):
        gpu = self.ctx.denoise_temporal(self.w, self.h, reset=reset, **self.dn)
        *cpu, self.history = dtl.oracle_denoise_temporal(self.rgb, self.aov["albedo"], self.aov["normal"], self.aov["hit_t"], self.cam, self.aov_params,
                                                        self.history, scene=self.scene, flags=self.flags, reset=reset, **self.dn)
        return gpu, tuple(cpu)

    def frame(self, cam, seed, reset=False):
        self.render(cam, seed)
        return self.denoise(reset)


def assert_same(gpu, cpu, what):
    bad = [int((g.view(np.uint32) != c.view(np.uint32)).sum()) for g, c in zip(gpu, cpu)]
    assert bad == [0, 0, 0], f"{what}: {bad[0]} pixels, {bad[1]} rgb floats and {bad[2]} history lengths differ from the restatement"


def run_sequence(ctx, kind, name="c1", lens=False, flags=0, w=W, h=H, frames=4, seed=10, **kw):
    seq = Sequence(ctx, w, h, flags=flags, **kw)
    lengths = []
    for i in range(frames):
        gpu, cpu = seq.frame(motion(kind, w, h, i, lens), seed + i, reset=i == 0)
        assert_same(gpu, cpu, f"{name} {kind} frame {i}")
        lengths.append(gpu[2])
        st = ctx.stats()
        assert st.kernel_launches == 2 + seq.dn.get("iterations", 5) and st.rays == 0 and st.device_ms > 0
    return lengths


@pytest.mark.parametrize("flags", [0, abi.FLAG_BVH, abi.FLAG_NO_JITTER], ids=["none", "bvh", "no_jitter"])
@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("kind", ["still", "pan", "translate", "rotate"])
@pytest.mark.parametrize("name", ["c1", "cloud", "mesh"])
def test_sequences_equal_the_restatement(gpu_ctx, name, kind, lens, flags):
    gpu_ctx.upload(scene_of(name))
    lengths = run_sequence(gpu_ctx, kind, name, lens, flags)
    assert lengths[-1].max() > 1.0, "no pixel kept any history"


@pytest.mark.parametrize("w,h", [(37, 23), (2, 64), (64, 2), (2, 2)])
def test_odd_sizes(gpu_ctx, w, h):
    scene, _ = scenes.rtiow_four_spheres(w, h)
    gpu_ctx.upload(scene)
    run_sequence(gpu_ctx, "translate", w=w, h=h)


@pytest.mark.parametrize("kw", [dict(alpha_color=0.5, alpha_moments=0.05, depth_tolerance=0.01, normal_cos=0.99, iterations=2, sigma_luminance=0.5),
                                dict(alpha_color=1.0, alpha_moments=1.0, depth_tolerance=1.0, normal_cos=-1.0, iterations=8, sigma_normal=7.0)])
def test_non_default_parameters(gpu_ctx, kw):
    scene, _ = scenes.rtiow_four_spheres(61, 45)
    gpu_ctx.upload(scene)
    run_sequence(gpu_ctx, "rotate", w=61, h=45, frames=5, **kw)


def test_full_size_c2_sequence(gpu_ctx):
    c = fs.CONFIGS["c2"]
    scene, cam = c["scene"](c["w"], c["h"])
    gpu_ctx.upload(scene)
    seq = Sequence(gpu_ctx, c["w"], c["h"], spp=2, aov_spp=2, depth=c["depth"])
    o, hor, ver, llc = (np.array(getattr(cam, k)[:], f32) for k in ("origin", "horizontal", "vertical", "lower_left_corner"))
    for i in range(4):
        shift = np.array([0.02 * i, 0.0, 0.01 * i], f32)
        gpu, cpu = seq.frame(cam_of(o + shift, hor, ver, llc + shift), 20 + i, reset=i == 0)
        assert_same(gpu, cpu, f"C2 frame {i}")


def test_first_call_and_reset_equal_denoise_and_still_camera_counts_calls(gpu_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    gpu_ctx.upload(scene)
    seq = Sequence(gpu_ctx, W, H, flags=abi.FLAG_NO_JITTER)  # fixed primary rays: the same surface point in every frame
    for i in range(5):
        seq.render(cam, 40 + i)
        plain = gpu_ctx.denoise(W, H)
        gpu, cpu = seq.denoise(reset=i in (0, 3))
        assert_same(gpu, cpu, f"frame {i}")
        if i in (0, 3):
            assert np.array_equal(gpu[0], plain[0]) and np.array_equal(gpu[1].view(np.uint32), plain[1].view(np.uint32))
        assert np.all(gpu[2] == (i + 1 if i < 3 else i - 2)), np.unique(gpu[2])


def test_pan_restarts_the_entering_columns(gpu_ctx):
    scene, _ = scenes.rtiow_four_spheres(W, H)
    gpu_ctx.upload(scene)
    k = 3
    seq = Sequence(gpu_ctx, W, H, flags=abi.FLAG_NO_JITTER)
    for i in range(4):
        gpu, cpu = seq.frame(motion("pan", W, H, i, step=k), 60 + i, reset=i == 0)
        assert_same(gpu, cpu, f"pan frame {i}")
        n = gpu[2]
        if i == 0:
            assert np.all(n == 1)
            continue
        assert np.all(n[:, W - k:] == 1), n[:, W - k:]
        # the rest follow their surface point: it left the frame or keeps growing (away from geometric edges)
        assert np.mean(n[:, :W - k] > 1) > 0.9, np.mean(n[:, :W - k] > 1)


def test_new_upload_or_size_drops_the_history(gpu_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    gpu_ctx.upload(scene)
    seq = Sequence(gpu_ctx, W, H, flags=abi.FLAG_NO_JITTER)
    seq.frame(cam, 1, reset=True)
    gpu, _ = seq.frame(cam, 2)
    assert np.all(gpu[2] == 2)
    gpu_ctx.upload(scene)                                          # same scene, new upload
    seq.scene += 1
    gpu, cpu = seq.frame(cam, 3)
    assert_same(gpu, cpu, "after an upload")
    assert np.all(gpu[2] == 1)
    gpu, _ = seq.frame(cam, 4)
    assert np.all(gpu[2] == 2)
    scene2, cam2 = scenes.rtiow_four_spheres(W + 3, H)
    other = Sequence(gpu_ctx, W + 3, H, flags=abi.FLAG_NO_JITTER)
    other.scene = seq.scene
    other.history = seq.history
    gpu, cpu = other.frame(cam2, 5)                                # another size
    assert_same(gpu, cpu, "after a size change")
    assert np.all(gpu[2] == 1)


def pt(w=W, h=H, **kw):
    kw.setdefault("spp", 4)
    kw.setdefault("seed", 2)
    return abi.make_params(w, h, mode=abi.MODE_PATHTRACE, max_depth=4, flags=abi.FLAG_NO_JITTER, **kw)


def test_refusals_change_nothing(built):
    ctx = abi.Context(0)
    try:
        scene, cam = scenes.rtiow_four_spheres(W, H)
        ctx.upload(scene)
        refused = []

        def refuse(match, **dn):
            with pytest.raises(abi.Rt3Error, match=match):
                ctx.denoise_temporal(dn.pop("w", W), dn.pop("h", H), **dn)
            refused.append(match)

        refuse("rt3_denoise_temporal needs a path-traced render")
        ctx.render(cam, pt())
        refuse("rt3_denoise_temporal needs an rt3_render_path_aovs")
        ctx.render_path_aovs(cam, pt())
        ctx.denoise_temporal(W, H, reset=True)                                    # frame A: history of length 1
        ctx.render(cam, pt(seed=3))
        ctx.render_path_aovs(cam, pt(seed=3))
        for bad, msg in ((dict(iterations=0), "iterations"), (dict(sigma_luminance=0.0), "sigma_luminance"), (dict(sigma_normal=2.5), "sigma_normal"),
                         (dict(alpha_color=0.0), "alpha_color"), (dict(alpha_color=1.5), "alpha_color"), (dict(alpha_moments=float("nan")), "alpha_moments"),
                         (dict(depth_tolerance=0.0), "depth_tolerance"), (dict(depth_tolerance=float("inf")), "depth_tolerance"),
                         (dict(normal_cos=1.01), "normal_cos"), (dict(normal_cos=float("nan")), "normal_cos")):
            refuse(f"rt3_denoise_temporal: {msg}", **bad)
        refuse("rt3_denoise_temporal: the last path-traced frame was", w=W + 1)
        ctx.render(cam, pt(seed=3, tile_rows=2, part_index=0, part_count=2))
        refuse("rt3_denoise_temporal: the path-traced render covers part")
        ctx.render(cam, pt(seed=3))
        ctx.render_path_aovs(abi.reference_camera(W, H, focal_length=1.5), pt(seed=3))
        refuse("rt3_denoise_temporal: the AOVs and the render used different cameras")
        ctx.render_path_aovs(cam, pt(seed=3, tile_rows=2, part_index=1, part_count=2))
        refuse("rt3_denoise_temporal: the AOVs cover part")
        ctx.render_path_aovs(cam, pt(seed=3))
        after = ctx.denoise_temporal(W, H)                                        # frame B on the history of frame A
        assert np.all(after[2] == 2), "a refused call changed the history"
        # the same two frames without the refusals in between
        ctx.render(cam, pt())
        ctx.render_path_aovs(cam, pt())
        ctx.denoise_temporal(W, H, reset=True)                                    # frame A
        ctx.render(cam, pt(seed=3))
        ctx.render_path_aovs(cam, pt(seed=3))
        clean = ctx.denoise_temporal(W, H)
        assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(after, clean))
        with pytest.raises(abi.Rt3Error, match="params is NULL"):
            ctx._check(ctx.lib.rt3_denoise_temporal(ctx.handle, None, None, None, None))
        assert len(refused) == 16
    finally:
        ctx.close()


def test_other_state_is_left_alone(gpu_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    gpu_ctx.upload(scene)
    k = 6
    first = gpu_ctx.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=k, max_depth=8, seed=5))
    aov = gpu_ctx.render_path_aovs(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=3, max_depth=8, seed=5))
    radiance = gpu_ctx.read_radiance(W, H)
    plain = gpu_ctx.denoise(W, H)
    for reset in (True, False, False):
        gpu_ctx.denoise_temporal(W, H, reset=reset)
    assert np.array_equal(gpu_ctx.read_radiance(W, H).view(np.uint32), radiance.view(np.uint32))
    again = gpu_ctx.denoise(W, H)
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(plain, again))
    aov2 = gpu_ctx.render_path_aovs(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=3, max_depth=8, seed=5))
    assert all(np.array_equal(aov[key].view(np.uint8), aov2[key].view(np.uint8)) for key in aov)
    more = gpu_ctx.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=k, max_depth=8, seed=5, flags=abi.FLAG_ACCUMULATE, first_sample=k))
    once = gpu_ctx.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=2 * k, max_depth=8, seed=5))
    assert np.array_equal(more, once) and not np.array_equal(first, once)


def quality(ctx, w, h, cams, spp=16):
    """PSNR (dB, packed 8-bit levels) at the last camera against a 4096-spp render of another seed: raw spp, raw 4 spp per
    frame, rt3_denoise of the last frame and rt3_denoise_temporal after every frame."""
    ref = ol.unpack_rgb(ctx.render(cams[-1], abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=4096, max_depth=50, seed=9999)))
    for i, cam in enumerate(cams):
        raw = ctx.render(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=50, seed=100 + i))
        ctx.render_path_aovs(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=50, seed=100 + i))
        temporal, _, _ = ctx.denoise_temporal(w, h, reset=i == 0)
    spatial, _ = ctx.denoise(w, h)
    raw_more = ctx.render(cams[-1], abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp * len(cams), max_depth=50, seed=500))
    q = {k: round(ol.psnr_levels(ol.unpack_rgb(f), ref), 2) for k, f in
         ((f"raw{spp}", raw), (f"raw{spp * len(cams)}", raw_more), ("denoise", spatial), ("temporal", temporal))}
    return q


def test_quality_still_camera(gpu_ctx):
    c = fs.CONFIGS["c1"]
    scene, cam = c["scene"](c["w"], c["h"])
    gpu_ctx.upload(scene)
    q = quality(gpu_ctx, c["w"], c["h"], [cam] * 4)
    print("C1 still, 4 x 16 spp, PSNR dB:", q)
    assert q["temporal"] > q["denoise"], q


def test_quality_slow_orbit(gpu_ctx):
    c = fs.CONFIGS["c1"]
    w, h = c["w"], c["h"]
    scene, cam = c["scene"](w, h)
    gpu_ctx.upload(scene)
    q = quality(gpu_ctx, w, h, [motion("orbit", w, h, i, base=cam) for i in range(8)])
    print("C1 slow orbit, 8 x 16 spp, PSNR dB:", q)
    assert q["temporal"] > q["denoise"], q


def test_host_backend(built):
    """CudaRenderer::denoise_temporal on one render, called four times: the first three equal CudaRenderer::denoise (no history,
    then a history equal to the new frame: c = e exactly, and the 7x7 variance below 4 frames); the fourth takes the
    moments' variance, 0 for a constant history, and so differs. A renderer on several devices refuses."""
    import hostlib
    from test_gpu_path_aovs import host_rtiow
    import path_aov_lib as pal
    w, h = 64, 36
    hs = host_rtiow(w, h, False)
    hs.render(w, h, focal=1.0)
    pal.host_path_aovs(hs, w, h, 5, focal=1.0)
    plain = dl.host_denoise(hs, w, h, focal=1.0)
    for i in range(4):
        got = dtl.host_denoise_temporal(hs, w, h, focal=1.0, reset=i == 0)
        same = np.array_equal(got[0], plain[0]) and np.array_equal(got[1].view(np.uint32), plain[1].view(np.uint32))
        assert same == (i < 3), i
    multi = host_rtiow(w, h, True)
    multi.render(w, h, focal=1.0)
    pal.host_path_aovs(multi, w, h, 5, focal=1.0)
    with pytest.raises(hostlib.HostError, match="one device"):
        dtl.host_denoise_temporal(multi, w, h, focal=1.0)
