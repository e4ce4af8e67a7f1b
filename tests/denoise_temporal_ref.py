"""Float64 reference of rt3_denoise_temporal's reprojection and accumulation (DESIGN.md 3.9) (TEST INFRASTRUCTURE).

Written from the formulas of DESIGN.md 3.9, not from the header's functions: numpy float64 throughout, the projection by
``np.linalg.solve``, true division. The demodulation, luminance, guide and 7x7 variance are tests/denoise_ref.py's.

``TEMPORAL_MUTATIONS`` names plausible wrong versions of single rules; ``temporal_step(..., mutation=name)`` applies one."""
import numpy as np

from denoise_ref import Taps, demodulate, guide, luminance, variance

TEMPORAL_MUTATIONS = {
    "motion_sign": "the previous position is (x, y) minus the motion instead of plus",
    "bilinear_swapped": "the bilinear weights of x and y are swapped",
    "alpha_no_floor": "alpha is 1/n without its floor alpha_color / alpha_moments",
    "depth_zp": "the depth test compares the tap's depth with z_p instead of |X - O_prev|",
    "no_weight_floor": "any positive used weight gives history, without the 0.01 floor",
    "miss_with_hit": "a miss takes history from hit taps (the miss agreement test dropped for misses)",
}


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
    ``variance_moments`` max(0, m2 - m1^2) and ``variance`` (from the moments from n >= 4, else the 7x7 estimate)."""
    assert mutation is None or mutation in TEMPORAL_MUTATIONS, mutation
    rgb, albedo, normal, depth, rays = (np.asarray(a, np.float64) for a in (rgb, albedo, normal, depth, rays))
    h, w = depth.shape
    e, _ = demodulate(rgb, albedo)
    L = luminance(e)
    nhat, z, miss = guide(normal, depth)
    sw = np.zeros((h, w))
    sc = np.zeros((h, w, 3))
    s1, s2, sn = np.zeros((h, w)), np.zeros((h, w)), np.zeros((h, w))
    near = np.zeros((h, w), bool)
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
                near |= inside & ~miss & ~mq & ((np.abs(dz) <= 4 * tau * ref_d) | (np.abs(cos) <= 4 * tau))
                near |= inside & prev["uncertain"][qyc, qxc]
                wu = np.where(use, wt, 0.0)
                sw += wu
                sc += wu[..., None] * prev["c"][qyc, qxc]
                s1 += wu * prev["m1"][qyc, qxc]
                s2 += wu * prev["m2"][qyc, qxc]
                sn += wu * prev["n"][qyc, qxc]
    floor = 0.0 if mutation == "no_weight_floor" else 0.01
    have = sw > floor
    near |= np.abs(sw - 0.01) <= 4 * tau
    with np.errstate(invalid="ignore", divide="ignore"):
        ch, h1, h2, nh = sc / sw[..., None], s1 / sw, s2 / sw, sn / sw
    n = np.where(have, nh + 1.0, 1.0)
    with np.errstate(divide="ignore"):
        ac = 1.0 / n if mutation == "alpha_no_floor" else np.maximum(alpha_color, 1.0 / n)
        am = 1.0 / n if mutation == "alpha_no_floor" else np.maximum(alpha_moments, 1.0 / n)
    c = np.where(have[..., None], ch + ac[..., None] * (e - ch), e)
    m1 = np.where(have, h1 + am * (L - h1), L)
    m2 = np.where(have, h2 + am * (L * L - h2), L * L)
    var_m = np.maximum(m2 - m1 * m1, 0.0)
    var_s, _ = variance(Taps(h, w, 3), (nhat, z, miss), luminance(c), sigma_depth, sigma_normal)
    hist = {"c": c, "m1": m1, "m2": m2, "n": n, "nhat": nhat, "z": z, "miss": miss, "camera": cam, "uncertain": near}
    return {"history": hist, "near_bound": near, "variance_moments": var_m, "variance": np.where(n >= 4, var_m, var_s)}
