"""The whole temporal call of the CPU restatement (tests/denoise_oracle.c) against the float64 reference
``denoise_temporal_ref.temporal_denoise``: steps 2-9 of DESIGN.md 3.9, every à-trous pass, the history length, the linear
rgb and the 8-bit frame, at every frame of 7-frame sequences. No GPU needed.

The restatement is stateless: each frame is re-run from the same carried history with 1..8 iterations, which gives every
pass. The tolerance, frame rule and hull bound are tests/test_denoise_reference.py's (tau = 2^-12, a floor of 10^-2 of the
image's largest value). Pixels the reference marks ``near_bound`` (a history test within tau of its bound, a fractional
length within 16 tau of 4, a variance that cancels by more than 2^12), and every pixel that later reads one, are held to
the hull bound only, and counted.

Inputs: the plane sequences of tests/test_denoise_temporal_cpu.py; an analytic scene of three spheres in front of a wall
under a sky (float64 ray-sphere depths and normals of the restatement's own jittered primary rays), translated and
rotated, so that silhouettes disocclude, the normal test rejects taps and misses lie next to hits; half-pixel pans whose
history positions fall in (-1, 0) and (W - 1, W); a sky of constant luminance (a moment variance of 0); 2xN and Nx2 frames,
the thinnest a render allows.

With the history length summed as sum w n / sum w (before the fix of rt3_dn_accumulate_px), taps that all carry n = 3
gave 3.9999998 for non-dyadic weights and the 7x7 branch of step 7: test_whole_lengths_stay_whole and the fourth frame of
the translated thin-lens plane sequence (4.5e-3 from the reference in its first pass) fail."""
import numpy as np
import pytest

import denoise_lib as dl
import denoise_temporal_ref as tref
from rt3_b200 import abi
from test_denoise_reference import TAU, compare, ill_conditioned, rel_error
from test_denoise_temporal_cpu import cam_arrays, case_frame, params, plane_scene, shifted, thin_lens

f32 = np.float32
ITERATIONS = 8   # every pass the call allows (RT3_DN_MAX_ITERATIONS)


# ---- inputs ----------------------------------------------------------------------------------------------------------------

SPHERES = [((-0.7, -0.1, -3.4), 0.7), ((0.55, -0.25, -2.8), 0.55), ((0.0, 0.5, -5.0), 1.0)]
WALL_Z, WALL_TOP = -6.0, 1.2


def sphere_scene(rays, seed, sky_level=None):
    """Radiance, albedo, normal and depth of three spheres in front of the wall z = -6 (up to y = 1.2) under a sky, hit by
    `rays` [H, W, 6] (origin, unit direction), in float64, returned as float32. The sky's radiance is noisy, or the
    constant `sky_level`."""
    o, d = rays[..., :3].astype(np.float64), rays[..., 3:].astype(np.float64)
    h, w = rays.shape[:2]
    n = np.zeros((h, w, 3))
    alb = np.ones((h, w, 3))
    tw = (WALL_Z - o[..., 2]) / d[..., 2]
    hit = (tw > 0) & (o[..., 1] + tw * d[..., 1] < WALL_TOP)
    t = np.where(hit, tw, np.inf)
    n[hit] = (0.0, 0.0, 1.0)
    alb[hit] = (0.6, 0.55, 0.45)
    for k, (c, r) in enumerate(SPHERES):
        oc = o - np.array(c)
        b = np.sum(oc * d, -1)
        disc = b * b - (np.sum(oc * oc, -1) - r * r)
        with np.errstate(invalid="ignore"):
            ts = -b - np.sqrt(disc)
        hit = (disc > 0) & (ts > 1e-4) & (ts < t)
        t = np.where(hit, ts, t)
        p = o + ts[..., None] * d
        n = np.where(hit[..., None], (p - np.array(c)) / r, n)
        alb = np.where(hit[..., None], np.array([(0.8, 0.3, 0.3), (0.3, 0.8, 0.4), (0.4, 0.5, 0.9)][k]), alb)
    rng = np.random.default_rng(seed)
    miss = np.isinf(t)
    shade = 0.3 + 0.7 * np.maximum(n @ np.array([0.3, 0.9, 0.3]), 0.0)
    rgb = alb * shade[..., None] * (1 + 0.4 * rng.uniform(-1, 1, (h, w, 3)))
    sky = 0.5 + 0.3 * d[..., 1:2] * np.array([0.6, 0.8, 1.0])
    sky = np.full((h, w, 3), sky_level) if sky_level is not None else sky * (1 + 0.2 * rng.uniform(-1, 1, (h, w, 3)))
    rgb = np.where(miss[..., None], sky, rgb)
    return tuple(a.astype(f32) for a in (rgb, alb, n, t))


def rotated(cam, a):
    """The camera turned by `a` radians about the vertical axis through its origin."""
    o, hor, ver, llc = cam_arrays(cam)
    R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    out = abi.make_camera(o, R @ hor, R @ ver, R @ (llc - o) + o)
    out.lens_radius, out.lens_u[:], out.lens_v[:] = cam.lens_radius, cam.lens_u[:], cam.lens_v[:]
    return out


def sphere_frame(kind, lens, i, w=61, h=45, sky_level=None):
    base = abi.reference_camera(w, h)
    if lens:
        thin_lens(base)
        base.lens_radius = 0.05
    cam = {"still": base, "translate": shifted(base, origin=(0.05 * i, 0.01 * i, 0), llc=(0.05 * i, 0.01 * i, 0)),
           "rotate": rotated(base, 0.015 * i)}[kind]
    p = params(w, h, seed=11 + i, flags=0)
    return cam, sphere_scene(dl.primary_rays(cam, p), seed=i, sky_level=sky_level), p


def pan_frame(step, i, w=23, h=13):
    """A pan of `step` pixels per frame on the plane under two sky rows: -0.5 puts column 0's history position in (-1, 0),
    +0.5 the last column's in (W - 1, W)."""
    base = thin_lens(abi.reference_camera(w, h))
    _, hor, _, _ = cam_arrays(base)
    cam = shifted(base, llc=step * i * hor / (w - 1))
    return cam, plane_scene(cam, w, h, sky_rows=2, seed=i), params(w, h, seed=3 + i, flags=0)


def strip_frame(w, h, i):
    """2xN and Nx2 frames (a render is at least 2x2): a plane, the camera translated along the strip (across it, each of
    its 2 pixels spans a third of the view, and the depth test between them would decide by a hair)."""
    base = abi.reference_camera(w, h)
    t = (0.03 * i, 0, 0) if w > h else (0, 0.03 * i, 0)
    cam = shifted(base, origin=t, llc=t)
    return cam, plane_scene(cam, w, h, seed=i), params(w, h, seed=5 + i, flags=0)


# id: frame i -> (camera, inputs, AOV params)
SEQUENCES = {
    **{f"plane_{kind}_{'lens' if lens else 'pinhole'}": (lambda i, kind=kind, lens=lens: case_frame(kind, lens, i))
       for kind, lens in [("still", False), ("pan", False), ("translate", True), ("dolly", False), ("dolly", True)]},
    "spheres_translate_pinhole": lambda i: sphere_frame("translate", False, i),
    "spheres_translate_lens": lambda i: sphere_frame("translate", True, i),
    "spheres_rotate_pinhole": lambda i: sphere_frame("rotate", False, i),
    "spheres_rotate_lens": lambda i: sphere_frame("rotate", True, i),
    "pan_left_half_pixel": lambda i: pan_frame(-0.5, i),
    "pan_right_half_pixel": lambda i: pan_frame(0.5, i),
    "strip_61x2": lambda i: strip_frame(61, 2, i),
    "strip_2x61": lambda i: strip_frame(2, 61, i),
}


# ---- the comparison ----------------------------------------------------------------------------------------------------------


def check_lengths(length, res, what):
    """The history length equals the reference's exactly where that is a whole number (unless a usable tap weighs within
    4 tau of 0), else within tau; pixels whose history depends on a test within tau of its bound are skipped. Returns the
    worst relative error."""
    n64, keep = res["n"], ~res["history"]["uncertain"]
    whole = keep & (n64 == np.round(n64)) & ~res["length_inexact"]
    bad = whole & (length != n64)
    assert not bad.any(), f"{what}: {int(bad.sum())} whole history lengths differ, e.g. {length[bad][:4]} for {n64[bad][:4]}"
    err = float((np.abs(length - n64) / n64)[keep].max(initial=0.0))
    assert err <= TAU, f"{what}: history length {err:.3g} from the reference"
    return err


def check_frame(passes, frame, rgb, length, hist32, ins, res, what):
    """One frame of a filter's output (every pass, the last call's frame, rgb and length) against the reference's
    ``temporal_denoise``. Returns (worst pass error, worst rgb error, worst length error, pixels held to the hull at each
    pass: the marks and every pixel that reads one by then)."""
    ill = ill_conditioned(res, len(passes))
    worst = compare(ins, passes, frame, what, skip_ill=True, res=res, hull_input=hist32, iterations=len(passes))
    err_n = check_lengths(length, res, what)
    err_rgb = rel_error(np.where(ill[-1][..., None], res["rgb"], rgb), res["rgb"])
    assert err_rgb <= TAU, f"{what}: rgb {err_rgb:.3g} from the reference"
    return worst, err_rgb, err_n, np.array([int(m.sum()) for m in ill])


def run(name, frames=7, mutation=None):
    """Runs sequence `name` through the restatement and the reference side by side. Yields per frame (restatement passes,
    frame, rgb, length, accumulated colour, inputs, reference result)."""
    hist = ref_hist = None
    for i in range(frames):
        cam, ins, p = SEQUENCES[name](i)
        passes = []
        for k in range(1, ITERATIONS + 1):
            frame, rgb, length, nxt = dl.oracle_denoise_temporal(*ins, cam, p, hist, iterations=k)
            passes.append(rgb.astype(np.float64) / np.maximum(ins[1].astype(np.float64), 1e-3))
        res = tref.temporal_denoise(*ins, dl.primary_rays(cam, p), cam, ref_hist, iterations=ITERATIONS, mutation=mutation)
        yield passes, frame, rgb, length, hist_colour(nxt), ins, res
        hist, ref_hist = nxt, res["history"]


def hist_colour(h):
    return h.col[..., :3].astype(np.float64)


class Held:
    """Worst errors and, per pass, the pixel-frames held to the hull bound over a sequence."""

    def __init__(self):
        self.worst, self.held, self.total = [0.0, 0.0, 0.0], 0, 0

    def add(self, errs, size):
        self.worst = [max(a, b) for a, b in zip(self.worst, errs[:3])]
        self.held = self.held + errs[3]
        self.total += size

    def share(self):
        return self.held / self.total

    def report(self, what):
        print(f"{what}: worst pass {self.worst[0]:.3g}, rgb {self.worst[1]:.3g}, length {self.worst[2]:.3g}; held to the hull per pass "
              + " ".join(f"{x:.0%}" for x in self.share()))


# Every other sequence is compared at every pass on at least three quarters of its pixel-frames. These are not: a history
# test within tau of its bound marks a few pixels a frame, the history carries the mark on, and the passes' footprints
# spread it; the spheres are held at 25-37 % of the pixel-frames in the first pass and entirely from the fourth, the 61x2
# strip at 27 % and 86 %, the dollied thin-lens plane at 2 % and 43 %. For them the first pass must compare half the
# pixel-frames. A mark that weighs how far its error can reach would narrow this; the reference does not have one.
SPREAD = {"spheres_translate_pinhole", "spheres_translate_lens", "spheres_rotate_pinhole", "spheres_rotate_lens", "strip_61x2", "plane_dolly_lens"}


@pytest.mark.parametrize("name", list(SEQUENCES))
def test_every_pass_against_the_reference(name):
    held = Held()
    for i, (passes, frame, rgb, length, c32, ins, res) in enumerate(run(name)):
        held.add(check_frame(passes, frame, rgb, length, c32, ins, res, f"{name} frame {i}"), length.size)
    held.report(name)
    share = held.share()
    assert share[0] < 0.5 if name in SPREAD else share.max() < 0.25, share


def test_constant_sky_is_held_to_the_hull():
    """A sky of constant radiance under albedo 1: L is the same in every frame, m2 - m1^2 cancels to 0 and the luminance stop
    is ill-conditioned; the reference marks those pixels and the restatement stays within its taps' hull there."""
    SEQUENCES["spheres_constant_sky"] = lambda i: sphere_frame("translate", True, i, sky_level=0.7)
    try:
        held = 0
        for i, (passes, frame, rgb, length, c32, ins, res) in enumerate(run("spheres_constant_sky")):
            check_frame(passes, frame, rgb, length, c32, ins, res, f"constant sky frame {i}")
            sky = np.isinf(ins[3])
            if i >= 3:
                assert sky.any() and res["near_bound"][sky & (res["n"] >= 4)].all()
            held += int(res["near_bound"].sum())
        assert held > 0
    finally:
        del SEQUENCES["spheres_constant_sky"]


# ---- whole lengths stay whole (the fix of rt3_dn_accumulate_px) -------------------------------------------------------------


def still_then_pan(dx, dy, w=27, h=19, sky=(0, 0, 0, 0)):
    """Three frames of a still thin-lens camera on the plane, then a pan of (dx, dy) pixels; frame i has `sky[i]` sky rows.
    Returns the restatement's per-frame (length, history) and the last frame's positions in the previous frame."""
    base = thin_lens(abi.reference_camera(w, h))
    _, hor, ver, _ = cam_arrays(base)
    hist, out = None, []
    for i in range(4):
        cam = base if i < 3 else shifted(base, llc=dx * hor / (w - 1) - dy * ver / (h - 1))
        ins = plane_scene(cam, w, h, sky_rows=sky[i], seed=i)
        p = params(w, h, seed=20 + i, flags=0)
        prev_cam = hist.camera if hist is not None else cam
        _, _, length, hist = dl.oracle_denoise_temporal(*ins, cam, p, hist)
        out.append((length, hist))
    rays = dl.primary_rays(cam, p).reshape(-1, 6)
    y, x = np.mgrid[0:h, 0:w]
    pos = dl.reproject(cam, prev_cam, w, h, np.stack([x, y], -1).reshape(-1, 2), rays, ins[3].reshape(-1)).reshape(h, w, 4)
    return out, pos, (cam, ins, p)


def test_whole_lengths_stay_whole():
    """A sub-pixel pan of (0.3, 0.1) pixels after three still frames: every used tap has n = 3 and weights that are not
    dyadic, for which sum w 3 / sum w rounds to 2.9999998 at some pixels in binary32. The length must be exactly 4, so that
    step 7 takes the moments' variance."""
    seq, pos, _ = still_then_pan(0.3, 0.1)
    assert [float(np.unique(length)[0]) for length, _ in seq[:3]] == [1.0, 2.0, 3.0]
    length = seq[3][0]
    inner = (pos[..., 0] > 0) & (pos[..., 0] < length.shape[1] - 1) & (pos[..., 1] > 0) & (pos[..., 1] < length.shape[0] - 1)
    assert inner.mean() > 0.8
    # the case bites: the plain weighted mean of four 3s is not 3 in binary32 at some of these pixels
    fx, fy = (pos[..., 0] - np.floor(pos[..., 0])).astype(f32), (pos[..., 1] - np.floor(pos[..., 1])).astype(f32)
    ws = [(f32(1) - fy) * (f32(1) - fx), (f32(1) - fy) * fx, fy * (f32(1) - fx), fy * fx]
    sw = sn = f32(0)
    for wt in ws:
        sw, sn = sw + wt, sn + wt * f32(3)
    assert ((sn / sw != f32(3)) & inner).any()
    assert np.all(length[inner] == 4.0), np.unique(length[inner])


def test_mixed_lengths_give_the_weighted_length():
    """Row 3 turns from sky into plane at frame 1 and restarts, so that after three still frames it holds n = 2 and the
    rows below n = 3; a vertical pan of 0.4 rows then mixes them. The length of every plane pixel is 1 + the bilinear mean
    of its used taps' lengths, from the positions the restatement computes, within 10^-6."""
    seq, pos, _ = still_then_pan(0.0, 0.4, sky=(4, 3, 3, 3))
    prev_len = seq[2][0]
    assert set(np.unique(prev_len[3:5])) == {2.0, 3.0}
    length = seq[3][0]
    h, w = length.shape
    px, py = pos[..., 0].astype(np.float64), pos[..., 1].astype(np.float64)
    x0, y0 = np.floor(px).astype(int), np.floor(py).astype(int)
    fx, fy = px - x0, py - y0
    sw = sn = 0.0
    for ty in (0, 1):
        for tx in (0, 1):
            wt = (fy if ty else 1 - fy) * (fx if tx else 1 - fx)
            qx, qy = np.clip(x0 + tx, 0, w - 1), np.clip(y0 + ty, 0, h - 1)
            ok = (wt > 0) & (x0 + tx >= 0) & (x0 + tx < w) & (y0 + ty >= 3) & (y0 + ty < h)   # rows 0-2 are sky: no tap for a hit
            sw = sw + np.where(ok, wt, 0.0)
            sn = sn + np.where(ok, wt * prev_len[qy, qx], 0.0)
    hits, have = np.arange(h)[:, None] >= 3, sw > 0.01
    want = 1.0 + sn / np.where(have, sw, 1.0)
    mixed = hits & have & (want > 3.0) & (want < 4.0)
    assert mixed.sum() >= w, "the pan mixes no lengths"
    err = np.abs(length - want)[hits & have].max()
    assert err <= 1e-6, err


# ---- mutations of steps 7-9 ---------------------------------------------------------------------------------------------------

# mutation: the sequence on which check_frame refuses the mutated reference (every pass of it compared: SPREAD excluded)
KILLS = {
    "moments_from_5": "plane_still_pinhole",
    "variance_of_e": "plane_translate_lens",
    "atrous_of_e": "plane_pan_pinhole",
    "m2_towards_m1sq": "plane_translate_lens",
    "history_first_pass": "plane_pan_pinhole",
}


def test_every_filter_mutation_has_a_case():
    assert sorted(KILLS) == sorted(tref.FILTER_MUTATIONS)
    assert not set(KILLS.values()) & SPREAD


@pytest.mark.parametrize("mutation", list(tref.FILTER_MUTATIONS))
def test_filter_mutation_is_refused(mutation):
    """The comparison itself, with its exclusions, refuses the reference with one rule of steps 7-9 made wrong, on a
    sequence that it passes unmutated (test_every_pass_against_the_reference)."""
    with pytest.raises(AssertionError) as refused:
        for i, (passes, frame, rgb, length, c32, ins, res) in enumerate(run(KILLS[mutation], mutation=mutation)):
            check_frame(passes, frame, rgb, length, c32, ins, res, f"{mutation} frame {i}")
    print(f"{mutation} on {KILLS[mutation]}: {str(refused.value).splitlines()[0]}")
