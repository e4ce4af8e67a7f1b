"""Float64 reference of rt3_denoise_temporal's reprojection and accumulation (DESIGN.md 3.9) (TEST INFRASTRUCTURE).

Written from the formulas of DESIGN.md 3.9, not from the header's functions: numpy float64 throughout, the projection by
``np.linalg.solve``, true division. The demodulation, luminance, guide and 7x7 variance are tests/denoise_ref.py's.

``TEMPORAL_MUTATIONS`` names plausible wrong versions of single rules of steps 2-6, ``FILTER_MUTATIONS`` of steps 7-9;
``temporal_step(..., mutation=name)`` and ``temporal_denoise(..., mutation=name)`` apply one.

``temporal_denoise`` is the whole call (steps 2-9): the history of ``temporal_step``, then the à-trous passes of
tests/denoise_ref.py over the accumulated colour, in the shape ``denoise_ref.denoise`` returns."""
import numpy as np

from denoise_ref import MIN_ALBEDO, Taps, atrous_passes, demodulate, guide, luminance, resolve, variance

TEMPORAL_MUTATIONS = {
    "motion_sign": "the previous position is (x, y) minus the motion instead of plus",
    "bilinear_swapped": "the bilinear weights of x and y are swapped",
    "alpha_no_floor": "alpha is 1/n without its floor alpha_color / alpha_moments",
    "depth_zp": "the depth test compares the tap's depth with z_p instead of |X - O_prev|",
    "no_weight_floor": "any positive used weight gives history, without the 0.01 floor",
    "miss_with_hit": "a miss takes history from hit taps (the miss agreement test dropped for misses)",
}

FILTER_MUTATIONS = {
    "moments_from_5": "the variance comes from the moments from n >= 5 instead of n >= 4",
    "variance_of_e": "the 7x7 estimate runs over this frame's e instead of the accumulated c",
    "atrous_of_e": "the à-trous passes run over this frame's e instead of the accumulated c",
    "m2_towards_m1sq": "m2 is blended towards m1^2 instead of L^2",
    "history_first_pass": "the history keeps the first à-trous output instead of the unfiltered c (SVGF's choice)",
}

MOMENT_FRAMES = 4.0


def _cam(cam):
    return [np.array(getattr(cam, k)[:], np.float64) for k in ("origin", "horizontal", "vertical", "lower_left_corner")]


def project(cam, X, miss, w, h):
    """proj(cam, X): (x', y', s) with X - O = s (llc - O) + a hor + b ver (a miss: X is the direction and replaces X - O),
    x' = a/s (W-1), y' = (H-1) - b/s (H-1)."""
    o, hor, ver, llc = _cam(cam)
    r = np.where(miss[..., None], X, X - o)
    M = np.stack([llc - o, hor, ver], axis=1)
    sab = np.linalg.solve(M, r.reshape(-1, 3).T).T.reshape(r.shape)
    s, a, b = sab[..., 0], sab[..., 1], sab[..., 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        return a / s * (w - 1), (h - 1) - b / s * (h - 1), s


def temporal_step(rgb, albedo, normal, depth, rays, cam, prev, alpha_color=0.2, alpha_moments=0.2, depth_tolerance=0.05, normal_cos=0.9,
                  sigma_depth=1.0, sigma_normal=128.0, tau=2.0 ** -12, mutation=None):
    """One call of rt3_denoise_temporal up to its variance, in float64, on [H, W, 3] radiance / albedo / normal, [H, W] depth,
    the [H, W, 6] primary rays (origin, unit direction) of the AOV call's sample, its camera and the previous step's
    ``history`` (None: none). Returns a dict: ``history`` (c, m1, m2, n, the guide, the camera and ``uncertain``, the pixels
    whose history depends on a test within ``tau`` of its bound), ``near_bound`` (that mask for this step),
    ``variance_moments`` max(0, m2 - m1^2), ``variance`` (from the moments from n >= 4, else the 7x7 estimate),
    ``cancellation`` the factor by which the chosen variance's subtraction magnifies rounding errors of its terms (m2 / var
    for the moments, denoise_ref.variance's for the 7x7 estimate), and ``near_moment_frames``, the pixels whose n is not
    a whole number, or may not be, but is within 16 ``tau`` of 4 (the branch of step 7 depends on its last bits), and
    ``length_inexact``, the pixels with a usable tap whose weight is within 4 ``tau`` of 0 (float32 may use it where
    float64 does not, or the reverse, so that a whole n need not be whole on both sides)."""
    assert mutation is None or mutation in TEMPORAL_MUTATIONS or mutation in FILTER_MUTATIONS, mutation
    rgb, albedo, normal, depth, rays = (np.asarray(a, np.float64) for a in (rgb, albedo, normal, depth, rays))
    h, w = depth.shape
    e, _ = demodulate(rgb, albedo)
    L = luminance(e)
    nhat, z, miss = guide(normal, depth)
    sw = np.zeros((h, w))
    sc = np.zeros((h, w, 3))
    s1, s2, sn, n0 = np.zeros((h, w)), np.zeros((h, w)), np.zeros((h, w)), np.zeros((h, w))
    near = np.zeros((h, w), bool)
    light = np.zeros((h, w), bool)
    if prev is not None and prev["c"].shape[:2] == (h, w):
        o, d = rays[..., :3], rays[..., 3:]
        with np.errstate(invalid="ignore"):
            X = np.where(miss[..., None], d, o + np.where(miss, 0.0, z)[..., None] * d)
        cx, cy, cs = project(cam, X, miss, w, h)
        px_, py_, ps = project(prev["camera"], X, miss, w, h)
        y, x = np.mgrid[0:h, 0:w]
        sign = -1.0 if mutation == "motion_sign" else 1.0
        px, py = x + sign * (px_ - cx), y + sign * (py_ - cy)
        ok = (cs > 0) & (ps > 0) & np.isfinite(px) & np.isfinite(py)
        px, py = np.where(ok, px, -10.0), np.where(ok, py, -10.0)
        dist = np.linalg.norm(X - _cam(prev["camera"])[0], axis=-1)
        x0, y0 = np.floor(px), np.floor(py)
        fx, fy = px - x0, py - y0
        if mutation == "bilinear_swapped":
            fx, fy = fy, fx
        tap_n = []
        for ty in (0, 1):
            for tx in (0, 1):
                wt = (fy if ty else 1 - fy) * (fx if tx else 1 - fx)
                qx, qy = x0.astype(np.int64) + tx, y0.astype(np.int64) + ty
                inside = ok & (wt > 0) & (qx >= 0) & (qx < w) & (qy >= 0) & (qy < h)
                qxc, qyc = np.clip(qx, 0, w - 1), np.clip(qy, 0, h - 1)
                zq, mq, nq = prev["z"][qyc, qxc], prev["miss"][qyc, qxc], prev["nhat"][qyc, qxc]
                ref_d = z if mutation == "depth_zp" else dist
                with np.errstate(invalid="ignore"):
                    dz = np.abs(zq - ref_d) - depth_tolerance * ref_d
                    cos = np.sum(nhat * nq, axis=-1) - normal_cos
                    geo = np.where(miss, mq | (mutation == "miss_with_hit"), ~mq & (dz <= 0) & (cos >= 0))
                use = inside & geo
                # a test within 4 tau of its bound decides the tap only where the other test passes or is as close
                near_z, near_n = np.abs(dz) <= 4 * tau * ref_d, np.abs(cos) <= 4 * tau
                near |= inside & ~miss & ~mq & ((near_z & ((cos >= 0) | near_n)) | (near_n & ((dz <= 0) | near_z)))
                near |= inside & prev["uncertain"][qyc, qxc]
                tap_n.append((use, wt, prev["n"][qyc, qxc]))
                wu = np.where(use, wt, 0.0)
                n0 = np.where(use & (sw == 0), prev["n"][qyc, qxc], n0)   # the first used tap's length
                sw += wu
                sc += wu[..., None] * prev["c"][qyc, qxc]
                s1 += wu * prev["m1"][qyc, qxc]
                s2 += wu * prev["m2"][qyc, qxc]
                sn += wu * (prev["n"][qyc, qxc] - n0)
        # a used tap whose weight is within 4 tau of 0 may be used on one side only: where its length differs from another
        # used tap's, n stays close but not equal
        lo, hi = np.full((h, w), np.inf), np.full((h, w), -np.inf)
        for use, wt, nq in tap_n:
            lo, hi = np.where(use, np.minimum(lo, nq), lo), np.where(use, np.maximum(hi, nq), hi)
        for use, wt, nq in tap_n:
            light |= use & (wt <= 4 * tau) & (lo != hi)
        # a position within 4 tau of a pixel boundary may pick other taps in float32 where the lengths around it differ
        # (an unchanged camera gives the same bits twice in both precisions: its whole positions pick the same taps)
        still = all(np.array_equal(a, b) for a, b in zip(_cam(cam), _cam(prev["camera"])))
        edge = ok & (((np.minimum(fx, 1 - fx) <= 4 * tau) & ~(still & (fx == 0))) | ((np.minimum(fy, 1 - fy) <= 4 * tau) & ~(still & (fy == 0))))
        rx, ry = np.clip(np.round(px), 0, w - 1).astype(np.int64), np.clip(np.round(py), 0, h - 1).astype(np.int64)
        taps = Taps(h, w, 1)
        nmax = np.max([taps.view(np.where(np.isfinite(prev["n"]), prev["n"], 0.0), dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1)], axis=0)
        nmin = np.min([np.where(taps.valid(dy, dx), taps.view(prev["n"], dy, dx), np.inf) for dy in (-1, 0, 1) for dx in (-1, 0, 1)], axis=0)
        light |= edge & (nmax[ry, rx] != nmin[ry, rx])
    floor = 0.0 if mutation == "no_weight_floor" else 0.01
    have = sw > floor
    near |= np.abs(sw - 0.01) <= 4 * tau
    with np.errstate(invalid="ignore", divide="ignore"):
        ch, h1, h2, nh = sc / sw[..., None], s1 / sw, s2 / sw, n0 + sn / sw
    n = np.where(have, nh + 1.0, 1.0)
    with np.errstate(divide="ignore"):
        ac = 1.0 / n if mutation == "alpha_no_floor" else np.maximum(alpha_color, 1.0 / n)
        am = 1.0 / n if mutation == "alpha_no_floor" else np.maximum(alpha_moments, 1.0 / n)
    c = np.where(have[..., None], ch + ac[..., None] * (e - ch), e)
    m1 = np.where(have, h1 + am * (L - h1), L)
    m2 = np.where(have, h2 + am * ((m1 * m1 if mutation == "m2_towards_m1sq" else L * L) - h2), L * L)
    var_m = np.maximum(m2 - m1 * m1, 0.0)
    var_s, canc_s = variance(Taps(h, w, 3), (nhat, z, miss), luminance(e if mutation == "variance_of_e" else c), sigma_depth, sigma_normal)
    moments = n >= (MOMENT_FRAMES + 1 if mutation == "moments_from_5" else MOMENT_FRAMES)
    with np.errstate(divide="ignore", invalid="ignore"):
        canc_m = np.where(m2 > 0, m2 / var_m, 1.0)
    hist = {"c": c, "m1": m1, "m2": m2, "n": n, "nhat": nhat, "z": z, "miss": miss, "camera": cam, "uncertain": near}
    return {"history": hist, "near_bound": near, "variance_moments": var_m, "variance": np.where(moments, var_m, var_s),
            "cancellation": np.where(moments, canc_m, canc_s), "length_inexact": light,
            "near_moment_frames": (np.abs(n - MOMENT_FRAMES) <= 16 * tau) & ((n != np.round(n)) | light), "e": e}


def temporal_denoise(rgb, albedo, normal, depth, rays, cam, prev, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0,
                     gamma=True, mutation=None, **temporal):
    """One call of rt3_denoise_temporal in float64 (steps 2-9), on temporal_step's inputs. Returns a dict in the shape of
    ``denoise_ref.denoise``: ``input`` the accumulated demodulated colour c the passes start from, ``passes``, ``rgb``,
    ``level``, ``frame`` and ``cancellation``, plus ``history`` (for the next call), ``n`` and ``near_bound``: the pixels
    whose history depends on a test within tau of its bound, whose n is fractional within 16 tau of 4, or whose variance
    cancels by more than 2^12. ``cancellation`` is +inf on the first two kinds, so that test_denoise_reference's
    ill_conditioned() holds them, and every pixel that reads them later, to the hull bound only."""
    assert mutation is None or mutation in TEMPORAL_MUTATIONS or mutation in FILTER_MUTATIONS, mutation
    step = temporal_step(rgb, albedo, normal, depth, rays, cam, prev, sigma_depth=sigma_depth, sigma_normal=sigma_normal, mutation=mutation, **temporal)
    hist = step["history"]
    g = (hist["nhat"], hist["z"], hist["miss"])
    c = step["e"] if mutation == "atrous_of_e" else hist["c"]
    passes = atrous_passes(c, step["variance"], g, iterations, sigma_luminance, sigma_normal, sigma_depth)
    if mutation == "history_first_pass":
        hist = {**hist, "c": passes[0]}
    out = passes[-1] * np.maximum(np.asarray(albedo, np.float64), MIN_ALBEDO)
    level, frame = resolve(out, gamma)
    # the 7x7 estimate reads the accumulated colour of its window: a pixel whose history is uncertain taints it
    h, w = step["near_bound"].shape
    taps = Taps(h, w, 3)
    window = np.any([taps.view(step["near_bound"], dy, dx) for dy in range(-3, 4) for dx in range(-3, 4)], axis=0)
    uncertain = step["near_bound"] | step["near_moment_frames"] | (window & (hist["n"] < MOMENT_FRAMES))
    cancellation = np.where(uncertain, np.inf, step["cancellation"])
    return {"input": c, "passes": passes, "rgb": out, "level": level, "frame": frame, "cancellation": cancellation, "history": hist,
            "n": hist["n"], "length_inexact": step["length_inexact"], "near_bound": uncertain | ~(cancellation <= 2.0 ** 12)}
