"""Float64 reference of the edge-avoiding à-trous denoiser (rt3_denoise, DESIGN.md 3.8) (TEST INFRASTRUCTURE).

Written from the formulas of DESIGN.md 3.8 and the top comment of include/rt3_denoise.h, not from the header's functions:
numpy float64 throughout, np.exp, np.power and true division, one shifted view and validity mask per tap offset. It is the
second, independent reference of the filter; tests/denoise_oracle.c shares the header's arithmetic with the kernels and so
cannot see a mistake in it.

``MUTATIONS`` names plausible wrong versions of single rules. ``denoise(..., mutation=name)`` applies one of them; the
tests use them to show that their inputs and tolerance tell a wrong filter from the right one."""
import numpy as np

MIN_ALBEDO = 1e-3
EPS_Z = 1e-6
EPS_L = 1e-10
LUMA = np.array([0.2126, 0.7152, 0.0722])
B3 = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16])
G3 = np.array([1 / 4, 1 / 2, 1 / 4])

MUTATIONS = {
    "clamp_border": "taps outside the image read the nearest edge pixel instead of being skipped",
    "reach_one": "x_z divides by sigma_z z_p for every tap, without the reach s max(|dx|, |dy|)",
    "variance_w": "the variance update sums w var_q instead of w^2 var_q",
    "g3x3_unweighted": "g3x3 drops its geometry weights w_z w_n",
    "b3_flat": "the spline is (1/8, 1/4, 1/4, 1/4, 1/8)",
    "no_centre_in_sum": "the centre tap is left out of sum w",
    "miss_depth_zero": "a miss is a hit at depth 0",
    "unnormalised_normals": "the normal guide is the mean normal as it is, not normalised",
    "step_linear": "pass i steps i + 1 pixels instead of 2^i",
    "luminance_of_input": "the luminance stop compares the luminance of the input, not of the current pass",
}


class Taps:
    """Shifted views of per-pixel arrays: ``view(a, dy, dx)[y, x] = a[y + dy, x + dx]``, and ``valid(dy, dx)``, the mask of
    the pixels whose tap lies inside the image. With ``clamp`` the taps read the nearest edge pixel and are all valid."""

    def __init__(self, h, w, reach, clamp=False):
        self.h, self.w, self.r, self.clamp = h, w, reach, clamp
        self.inside = np.ones((h, w), bool)
        self.padded = {}

    def view(self, a, dy, dx):
        key = id(a)
        if key not in self.padded:
            pad = ((self.r, self.r), (self.r, self.r)) + ((0, 0),) * (a.ndim - 2)
            self.padded[key] = (a, np.pad(a, pad, mode="edge" if self.clamp else "constant"))
        p = self.padded[key][1]
        return p[self.r + dy:self.r + dy + self.h, self.r + dx:self.r + dx + self.w]

    def valid(self, dy, dx):
        return self.view(self.inside, dy, dx)


def demodulate(rgb, albedo):
    d = np.maximum(albedo, MIN_ALBEDO)
    return rgb / d, d


def luminance(e):
    return e @ LUMA


def guide(normal, depth, mutation=None):
    """(n^, z, miss): the normalised normal (0 where |n| = 0), the depth and the miss mask (depth +inf)."""
    miss = np.isposinf(depth)
    if mutation == "unnormalised_normals":
        nhat = normal.copy()
    else:
        length = np.linalg.norm(normal, axis=-1, keepdims=True)  # float64: no float32 normal over- or underflows here
        nhat = normal / np.where(length > 0, length, 1.0)
    z = depth.copy()
    if mutation == "miss_depth_zero":
        z[miss] = 0.0
        miss = np.zeros_like(miss)
    return nhat, z, miss


def geometry(taps, g, dy, dx, reach, sigma_z, sigma_n):
    """(x_z, w_n, linked) of the tap at offset (dy, dx) seen from every pixel: linked is False where exactly one of p and q
    is a miss (the tap's weight is 0) or where q lies outside the image; two misses give x_z = 0 and w_n = 1."""
    nhat, z, miss = g
    nq, zq, mq = taps.view(nhat, dy, dx), taps.view(z, dy, dx), taps.view(miss, dy, dx)
    both = miss & mq
    linked = taps.valid(dy, dx) & (miss == mq)
    with np.errstate(invalid="ignore", over="ignore"):
        x_z = np.where(miss | mq, 0.0, np.abs(z - zq) / (sigma_z * z * reach + EPS_Z))
    cos = np.maximum(np.sum(nhat * nq, axis=-1), 0.0)
    w_n = np.where(both, 1.0, np.power(cos, sigma_n))
    return x_z, w_n, linked


def variance(taps, g, lum, sigma_z, sigma_n, mutation=None):
    """max(0, E[L^2] - E[L]^2) over 7x7, weights w_z w_n at reach max(|dx|, |dy|), the centre 1."""
    sw = np.zeros(lum.shape)
    m1 = np.zeros(lum.shape)
    m2 = np.zeros(lum.shape)
    for dy in range(-3, 4):
        for dx in range(-3, 4):
            if dy == 0 and dx == 0:
                wt = np.ones(lum.shape)
            else:
                reach = 1 if mutation == "reach_one" else max(abs(dx), abs(dy))
                x_z, w_n, linked = geometry(taps, g, dy, dx, reach, sigma_z, sigma_n)
                wt = np.where(linked, w_n * np.exp(-x_z), 0.0)
            lq = taps.view(lum, dy, dx)
            sw += wt
            m1 += wt * lq
            m2 += wt * lq * lq
    var = np.maximum(m2 / sw - (m1 / sw) ** 2, 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        cancellation = np.where(m2 > 0, (m2 / sw) / var, 1.0)
    return var, cancellation


def g3x3(taps, g, var, sigma_z, sigma_n, mutation=None):
    """The 3x3 (1/4, 1/2, 1/4) blur of the variance at step 1, weighted by w_z w_n (reach 1) and normalised."""
    gs = np.zeros(var.shape)
    gv = np.zeros(var.shape)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            h = G3[dy + 1] * G3[dx + 1]
            if dy == 0 and dx == 0:
                wt = np.full(var.shape, h)
            elif mutation == "g3x3_unweighted":
                wt = np.where(taps.valid(dy, dx), h, 0.0)
            else:
                x_z, w_n, linked = geometry(taps, g, dy, dx, 1, sigma_z, sigma_n)
                wt = np.where(linked, h * w_n * np.exp(-x_z), 0.0)
            gs += wt
            gv += wt * taps.view(var, dy, dx)
    return gv / gs


def atrous_pass(e, var, lum_stop, g, step, sigma_l, sigma_z, sigma_n, mutation=None):
    """One pass at step ``step``: 5x5 taps at offsets step (dx, dy), w = h_y h_x w_n exp(-(x_z + x_l)), the centre h_2 h_2.
    Returns (the weighted mean of e, the variance sum w^2 var_q / (sum w)^2)."""
    h, w = var.shape
    taps = Taps(h, w, max(2 * step, 1), clamp=mutation == "clamp_border")
    b3 = np.array([1 / 8, 1 / 4, 1 / 4, 1 / 4, 1 / 8]) if mutation == "b3_flat" else B3
    l_den = sigma_l * np.sqrt(g3x3(taps, g, var, sigma_z, sigma_n, mutation)) + EPS_L
    sw = np.zeros((h, w))
    se = np.zeros((h, w, 3))
    sv = np.zeros((h, w))
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            hyx = b3[dy + 2] * b3[dx + 2]
            if dy == 0 and dx == 0:
                wt = np.full((h, w), hyx)
            else:
                reach = 1 if mutation == "reach_one" else step * max(abs(dx), abs(dy))
                x_z, w_n, linked = geometry(taps, g, dy * step, dx * step, reach, sigma_z, sigma_n)
                x_l = np.abs(lum_stop - taps.view(lum_stop, dy * step, dx * step)) / l_den
                with np.errstate(invalid="ignore"):
                    wt = np.where(linked, hyx * w_n * np.exp(-(x_z + x_l)), 0.0)
            if not (dy == 0 and dx == 0 and mutation == "no_centre_in_sum"):
                sw += wt
            se += wt[..., None] * taps.view(e, dy * step, dx * step)
            sv += (wt if mutation == "variance_w" else wt * wt) * taps.view(var, dy * step, dx * step)
    with np.errstate(invalid="ignore", divide="ignore"):
        return se / sw[..., None], sv / (sw * sw)


def resolve(rgb, gamma=True):
    """resolve_kernel's 8-bit frame of linear rgb: (levels before rounding [H, W, 3], packed frame [H, W] uint32). sqrt for
    the gamma, clamp to [0, 1] (NaN -> 0), times 255, rounded half away from zero."""
    v = np.sqrt(np.maximum(rgb, 0.0)) if gamma else rgb
    level = np.nan_to_num(np.clip(v, 0.0, 1.0), nan=0.0) * 255.0
    ch = np.floor(level + 0.5).astype(np.uint32)
    frame = (ch[..., 0] << 24) | (ch[..., 1] << 16) | (ch[..., 2] << 8) | np.uint32(0xFF)
    return level, frame


def denoise(rgb, albedo, normal, depth, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0, gamma=True, mutation=None):
    """rt3_denoise in float64 on [H, W, 3] radiance / albedo / normal and [H, W] depth (+inf on a miss).

    Returns a dict: ``input`` the demodulated radiance, ``passes`` the demodulated output of every pass, ``rgb`` the final
    linear radiance, ``level`` its 8-bit level before rounding, ``frame`` the packed frame, and ``cancellation`` E[L^2] / var
    of the 7x7 variance: the factor by which E[L^2] - E[L]^2 magnifies rounding errors of its terms."""
    assert mutation is None or mutation in MUTATIONS, mutation
    rgb, albedo, normal, depth = (np.asarray(a, np.float64) for a in (rgb, albedo, normal, depth))
    h, w = depth.shape
    e0, d = demodulate(rgb, albedo)
    g = guide(normal, depth, mutation)
    var, cancellation = variance(Taps(h, w, 3, clamp=mutation == "clamp_border"), g, luminance(e0), sigma_z=sigma_depth, sigma_n=sigma_normal,
                                 mutation=mutation)
    e = e0
    passes = []
    for i in range(iterations):
        step = i + 1 if mutation == "step_linear" else 2 ** i
        lum_stop = luminance(e0 if mutation == "luminance_of_input" else e)
        e, var = atrous_pass(e, var, lum_stop, g, step, sigma_luminance, sigma_depth, sigma_normal, mutation)
        passes.append(e)
    out = e * d
    level, frame = resolve(out, gamma)
    return {"input": e0, "passes": passes, "rgb": out, "level": level, "frame": frame, "cancellation": cancellation}
