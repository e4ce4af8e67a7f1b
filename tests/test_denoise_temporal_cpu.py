"""rt3_denoise_temporal without a GPU: the header's reprojection and accumulation (include/rt3_denoise.h) through the CPU
restatement (tests/denoise_temporal_oracle.c) on hand-checkable cases, against the float64 reference (tests/denoise_temporal_ref.py), and
with single-rule mutations of that reference; the parameter checks; the ABI; the new kernels' resources."""
import ctypes as C
import re
import shutil
import subprocess

import numpy as np
import pytest

import denoise_lib as dl
import denoise_temporal_lib as dtl
import denoise_temporal_ref as tref
from rt3_b200 import abi

f32 = np.float32
TAU = 2.0 ** -12


def params(w, h, seed=1, flags=abi.FLAG_NO_JITTER):
    return abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=1, max_depth=1, seed=seed, flags=flags)


def thin_lens(cam):
    cam.lens_radius = 0.1
    cam.lens_u[:] = [1, 0, 0]
    cam.lens_v[:] = [0, 1, 0]
    return cam


def cam_arrays(cam):
    return [np.array(getattr(cam, k)[:], np.float64) for k in ("origin", "horizontal", "vertical", "lower_left_corner")]


def shifted(cam, origin=(0, 0, 0), llc=(0, 0, 0)):
    o, hor, ver, c = cam_arrays(cam)
    out = abi.make_camera(o + origin, hor, ver, c + llc)
    out.lens_radius, out.lens_u[:], out.lens_v[:] = cam.lens_radius, cam.lens_u[:], cam.lens_v[:]
    return out


def plane_scene(cam, w, h, plane_z=-3.0, sky_rows=0, seed=0):
    """Per-pixel inputs of a camera looking at the plane z = plane_z (normal +z, albedo 0.5), the top `sky_rows` rows misses:
    (rgb, albedo, normal, depth) with depth along the unit direction of the unjittered pinhole ray."""
    o, hor, ver, llc = cam_arrays(cam)
    y, x = np.mgrid[0:h, 0:w]
    u, v = x / (w - 1), (h - 1 - y) / (h - 1)
    d = llc + u[..., None] * hor + v[..., None] * ver - o
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    depth = (plane_z - o[2]) / d[..., 2]
    rng = np.random.default_rng(seed)
    rgb = rng.uniform(0.1, 0.6, (h, w, 3))
    albedo = np.full((h, w, 3), 0.5)
    normal = np.broadcast_to([0.0, 0.0, 1.0], (h, w, 3)).copy()
    depth[:sky_rows] = np.inf
    normal[:sky_rows] = 0.0
    albedo[:sky_rows] = 1.0
    return rgb.astype(f32), albedo.astype(f32), normal.astype(f32), depth.astype(f32)


def rays_of(cam, w, h):
    """Unit pinhole rays through the pixel centres, float32: [h * w, 6] and the pixel coordinates [h * w, 2]."""
    o, hor, ver, llc = cam_arrays(cam)
    y, x = np.mgrid[0:h, 0:w]
    d = llc + (x / (w - 1))[..., None] * hor + ((h - 1 - y) / (h - 1))[..., None] * ver - o
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    rays = np.concatenate([np.broadcast_to(o, d.shape), d], -1).reshape(-1, 6)
    return rays.astype(f32), np.stack([x, y], -1).reshape(-1, 2).astype(f32)


@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
def test_unchanged_camera_maps_every_pixel_to_itself(lens):
    w, h = 23, 17
    cam = abi.reference_camera(w, h)
    if lens:
        thin_lens(cam)
    rays, xy = rays_of(cam, w, h)
    rng = np.random.default_rng(1)
    rays[:, :3] += rng.normal(0, 0.05, (len(rays), 3)).astype(f32)            # lens offsets
    depth = rng.uniform(0.5, 50, len(rays)).astype(f32)
    depth[::7] = np.inf
    pos = dtl.reproject(cam, cam, w, h, xy, rays, depth)
    assert np.all(pos[:, 3] == 1)
    assert np.array_equal(pos[:, :2], xy)


@pytest.mark.parametrize("k", [1.0, 2.5, -3.0])
def test_image_plane_pan_moves_by_k(k):
    w, h = 31, 19
    prev = abi.reference_camera(w, h)
    _, hor, _, _ = cam_arrays(prev)
    cur = shifted(prev, llc=k * hor / (w - 1))
    rays, xy = rays_of(cur, w, h)
    depth = np.random.default_rng(2).uniform(1, 20, len(rays)).astype(f32)
    depth[::5] = np.inf
    pos = dtl.reproject(cur, prev, w, h, xy, rays, depth)
    assert np.all(pos[:, 3] == 1)
    assert np.max(np.abs(pos[:, 0] - (xy[:, 0] + k))) < 1e-3
    assert np.max(np.abs(pos[:, 1] - xy[:, 1])) < 1e-3


def test_point_behind_the_previous_camera_has_no_history():
    w, h = 9, 7
    cur = abi.reference_camera(w, h)
    prev = shifted(cur, origin=(0, 0, -10), llc=(0, 0, -10))                  # 10 units further along -z, looking the same way
    rays, xy = rays_of(cur, w, h)
    pos = dtl.reproject(cur, prev, w, h, xy, rays, np.full(len(rays), 1.0, f32))  # points near z = -1: behind the previous camera
    assert np.all(pos[:, 3] == 0)


def run(frames, w, h, **kw):
    """Runs the restatement over [(camera, inputs, reset)], returns the (frame, rgb, length, history) of every call."""
    hist, out = None, []
    for cam, ins, reset in frames:
        res = dtl.oracle_denoise_temporal(*ins, cam, params(w, h), hist, reset=reset, **kw)
        hist = res[3]
        out.append(res)
    return out


@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
def test_first_frame_equals_denoise(lens):
    w, h = 29, 21
    cam = abi.reference_camera(w, h)
    if lens:
        thin_lens(cam)
    ins = plane_scene(cam, w, h, sky_rows=5)
    frame, rgb, length, _ = run([(cam, ins, False)], w, h)[0]
    want = dl.oracle_denoise(*ins)
    assert np.array_equal(frame, want[0]) and np.array_equal(rgb.view(np.uint32), want[1].view(np.uint32))
    assert np.all(length == 1)


def test_still_camera_counts_calls_and_alpha_follows_one_over_n_to_its_floor():
    w, h = 12, 9
    cam = abi.reference_camera(w, h)
    rgb, albedo, normal, depth = plane_scene(cam, w, h, sky_rows=2)
    frames = [(cam, (rgb * f32(1 + i), albedo, normal, depth), False) for i in range(8)]
    res = run(frames, w, h, alpha_color=0.2, alpha_moments=0.3)
    e = [(rgb * f32(1 + i)) / np.maximum(albedo, f32(1e-3)) for i in range(8)]
    c = e[0].astype(np.float64)
    for i, (_, _, length, hist) in enumerate(res):
        assert np.all(length == i + 1)
        if i:
            alpha = max(0.2, 1.0 / (i + 1))                                       # 1/2, 1/3, 1/4, then the floor 0.2
            c = c + alpha * (e[i] - c)
        assert np.allclose(hist.col[..., :3], c, rtol=1e-5), i


def test_misses_never_take_history_from_hits():
    w, h = 10, 8
    cam = abi.reference_camera(w, h)
    a = plane_scene(cam, w, h, sky_rows=3)
    b = plane_scene(cam, w, h, sky_rows=5, seed=1)                            # rows 3, 4 turn from hits into misses
    c = plane_scene(cam, w, h, sky_rows=1, seed=2)                            # rows 1..4 turn from misses into hits
    res = run([(cam, a, False), (cam, b, False), (cam, c, False)], w, h)
    assert np.all(res[1][2][3:5] == 1) and np.all(res[1][2][:3] == 2) and np.all(res[1][2][5:] == 2)
    assert np.all(res[2][2][1:5] == 1) and np.all(res[2][2][:1] == 3) and np.all(res[2][2][5:] == 3)


def tap_case(w, h, depth_scale=1.0, normal=None, **kw):
    cam = abi.reference_camera(w, h)
    a = plane_scene(cam, w, h)
    b = list(plane_scene(cam, w, h, seed=1))
    b[3] = (b[3] * f32(depth_scale)).astype(f32)
    if normal is not None:
        b[2] = np.broadcast_to(np.asarray(normal, f32), b[2].shape).copy()
    return run([(cam, a, False), (cam, tuple(b), False)], w, h, **kw)[1][2]


def test_depth_test_applies_just_inside_and_outside_its_bound():
    # the history's depth is z, the new surface point lies at z * s: |z - z s| <= tol z s  <=>  |1 - s| <= tol s
    tol = 0.05
    assert np.all(tap_case(8, 6, 1.0 / (1 - tol) * (1 - 1e-3), depth_tolerance=tol) == 2)   # just inside
    assert np.all(tap_case(8, 6, 1.0 / (1 - tol) * (1 + 1e-3), depth_tolerance=tol) == 1)   # just outside
    assert np.all(tap_case(8, 6, 1.0 / (1 + tol) * (1 + 1e-3), depth_tolerance=tol) == 2)
    assert np.all(tap_case(8, 6, 1.0 / (1 + tol) * (1 - 1e-3), depth_tolerance=tol) == 1)


def test_normal_test_applies_just_inside_and_outside_its_bound():
    for cos, want in ((0.9 + 1e-3, 2), (0.9 - 1e-3, 1)):
        n = [np.sqrt(1 - cos * cos), 0.0, cos]                                 # n^_p . (0, 0, 1) = cos
        assert np.all(tap_case(8, 6, normal=n, normal_cos=0.9) == want), cos


def test_weight_floor_applies_just_inside_and_outside():
    # a pan of 1 - f pixels: the last column's history is the tap at W - 1 with weight f (the other tap is outside)
    w, h = 16, 4
    prev = abi.reference_camera(w, h)
    _, hor, _, _ = cam_arrays(prev)
    for f, want in ((0.0105, 2), (0.0095, 1)):
        cur = shifted(prev, llc=(1 - f) * hor / (w - 1))
        # the wide view's plane recedes 10 % over that last pixel: a loose depth test, so that only the weight decides
        res = run([(prev, plane_scene(prev, w, h), False), (cur, plane_scene(cur, w, h, seed=1), False)], w, h, depth_tolerance=0.5)
        assert np.all(res[1][2][:, -1] == want), (f, res[1][2][:, -1])


def test_reset_and_size_change_drop_the_history():
    w, h = 10, 8
    cam = abi.reference_camera(w, h)
    ins = plane_scene(cam, w, h)
    res = run([(cam, ins, False), (cam, ins, False), (cam, ins, True), (cam, ins, False)], w, h)
    assert [float(r[2].max()) for r in res] == [1, 2, 1, 2]
    cam2 = abi.reference_camera(w + 1, h)
    big = dtl.oracle_denoise_temporal(*plane_scene(cam2, w + 1, h), cam2, params(w + 1, h), res[-1][3])
    assert np.all(big[2] == 1)


@pytest.mark.parametrize("bad,msg", [
    (dict(alpha_color=0.0), "alpha_color"), (dict(alpha_color=1.0001), "alpha_color"), (dict(alpha_color=float("nan")), "alpha_color"),
    (dict(alpha_moments=-0.1), "alpha_moments"), (dict(depth_tolerance=0.0), "depth_tolerance"), (dict(depth_tolerance=float("inf")), "depth_tolerance"),
    (dict(normal_cos=-1.5), "normal_cos"), (dict(normal_cos=float("nan")), "normal_cos"), (dict(iterations=0), "iterations"),
    (dict(sigma_normal=0.5), "sigma_normal")])
def test_invalid_parameters_are_refused_with_a_message(bad, msg):
    got = dtl.check_temporal_params(width=8, height=8, **bad)
    assert got is not None and got.startswith(msg), got


def test_valid_parameter_edges_are_accepted():
    for ok in (dict(), dict(alpha_color=1.0, alpha_moments=1.0), dict(normal_cos=-1.0), dict(normal_cos=1.0), dict(depth_tolerance=1e30)):
        assert dtl.check_temporal_params(width=8, height=8, **ok) is None, ok


# ---- the float64 reference ---------------------------------------------------------------------------------------------

def sequence_case(kind, lens, frames, w=27, h=19):
    """Yields (restatement history, reference step) of a sequence on a wavy plane under a sky whose lower edge moves by a
    row every other frame, jittered rays, and the camera `still`, panned by 0.995 px per frame (the last column's only
    tap then weighs 0.005, under the 0.01 floor), translated sideways and up, or dollied forward."""
    base = abi.reference_camera(w, h)
    if lens:
        thin_lens(base)
    _, hor, _, _ = cam_arrays(base)
    hist = ref_hist = None
    for i in range(frames):
        cam = {"still": base, "pan": shifted(base, llc=0.995 * i * hor / (w - 1)),
               "translate": shifted(base, origin=(0.04 * i, 0.01 * i, 0), llc=(0.04 * i, 0.01 * i, 0)),
               "dolly": shifted(base, origin=(0, 0, -0.25 * i), llc=(0, 0, -0.25 * i))}[kind]
        ins = plane_scene(cam, w, h, sky_rows=4 + i % 2, seed=i)
        ins = (ins[0], ins[1], ins[2], (ins[3] * f32(1 + 0.02 * np.sin(np.arange(w) / 3.0))).astype(f32))
        p = params(w, h, seed=7 + i, flags=0)
        _, _, _, hist = dtl.oracle_denoise_temporal(*ins, cam, p, hist)
        r = yield hist, ins, dtl.primary_rays(cam, p), cam, ref_hist
        ref_hist = r["history"]


def run_reference(kind, lens, frames, mutation=None):
    out = []
    gen = sequence_case(kind, lens, frames)
    item = next(gen)
    while True:
        hist, ins, rays, cam, ref_hist = item
        r = tref.temporal_step(*ins, rays, cam, ref_hist, mutation=mutation)
        out.append((hist, r))
        try:
            item = gen.send(r)
        except StopIteration:
            return out


def rel_err(a32, a64):
    return np.abs(a32 - a64) / np.maximum(np.abs(a64), 1e-2 * max(np.abs(a64).max(), 1e-30))


CASES = [("still", False), ("pan", False), ("translate", True), ("dolly", False), ("dolly", True)]


@pytest.mark.parametrize("kind,lens", CASES)
def test_restatement_matches_the_float64_reference(kind, lens):
    excluded = total = 0
    for i, (hist, r) in enumerate(run_reference(kind, lens, 7)):
        keep = ~r["near_bound"]
        excluded += int((~keep).sum())
        total += keep.size
        rh = r["history"]
        assert rel_err(hist.col[..., 3], rh["n"])[keep].max() <= TAU, i
        assert rel_err(hist.col[..., :3], rh["c"])[keep].max() <= TAU, i
        assert rel_err(hist.mom[..., 0], rh["m1"])[keep].max() <= TAU, i
        assert rel_err(hist.mom[..., 1], rh["m2"])[keep].max() <= TAU, i
    assert excluded < total / 4, (excluded, total)
    print(f"{kind} lens={lens}: {excluded} of {total} pixel-frames within tau of a bound, excluded")


@pytest.mark.parametrize("mutation", list(tref.TEMPORAL_MUTATIONS))
def test_mutations_are_far_from_the_restatement(mutation):
    worst = 0.0
    for kind, lens in CASES:
        for hist, r in run_reference(kind, lens, 7, mutation):
            rh = r["history"]
            worst = max(worst, rel_err(hist.col[..., :3], rh["c"]).max(), np.abs(hist.col[..., 3] - rh["n"]).max())
    assert worst > 10 * TAU, f"{mutation}: at most {worst} from the restatement"


# ---- ABI and resources ------------------------------------------------------------------------------------------------

def test_abi_symbol_and_layout(built):
    assert "rt3_denoise_temporal" in abi.EXPORTED_SYMBOLS
    assert hasattr(abi.load_core(), "rt3_denoise_temporal")
    T = abi.DenoiseTemporalParams
    assert C.sizeof(T) == 44
    assert [getattr(T, f).offset for f in ("filter", "alpha_color", "alpha_moments", "depth_tolerance", "normal_cos", "reset")] == [0, 24, 28, 32, 36, 40]
    p = abi.denoise_temporal_params()
    assert (p.alpha_color, p.alpha_moments, p.depth_tolerance, p.normal_cos, p.reset) == (f32(0.2), f32(0.2), f32(0.05), f32(0.9), 0)
    assert (p.filter.iterations, p.filter.sigma_luminance, p.filter.sigma_normal, p.filter.sigma_depth) == (5, 4.0, 128.0, 1.0)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
@pytest.mark.parametrize("needle", ["denoise_temporal_kernel", "denoise_temporal_variance_kernel"])
def test_new_kernels_keep_to_registers(built, needle):
    text = subprocess.run(["cuobjdump", "-res-usage", abi.CORE_LIB_PATH], check=True, capture_output=True, text=True).stdout
    found = [(m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))) for m in
             re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", text) if re.search(rf"\d{needle}", m.group(1))]
    assert len(found) == 1, found
    name, reg, stack, local = found[0]
    assert local == 0 and stack == 0, f"{name}: {local} bytes of local memory, {stack} bytes of stack"
    assert reg <= 64, f"{name}: {reg} registers"
