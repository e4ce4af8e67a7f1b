"""The denoiser's CPU restatement (tests/denoise_oracle.c, the arithmetic of include/rt3_denoise.h) against the independent
float64 reference tests/denoise_ref.py. No GPU needed.

The GPU tests pin the kernels bit for bit to the restatement, but both call the same header, so a mistake in the header
is on both sides of that comparison. These tests compare the header's filter with the formulas of DESIGN.md 3.8 evaluated in
float64: the primitives against libm, every pass of the filter on synthetic and rendered inputs, the convex-hull bound of
every pass, the 8-bit frame, and symmetries of the whole filter. For each mutation of the reference (one rule made wrong,
``denoise_ref.MUTATIONS``) a case of this file tells it from the restatement by more than 10 tau (``KILLS``).

Tolerance: the demodulated channels of every pass by ``|e32 - e64| / max(|e64|, f)``, f = 10^-2 times the largest |e64| of the
image, at most tau = 2^-12 (times sigma_n / 128 above 128: the normal power multiplies the float32 error of the dot product by
sigma_n). The worst value measured per case is in CASES.

Sabotage checks of the header, one at a time, each rebuilt (the restatement is compiled from the header on first use):
  - B3 centre 0.375 -> 0.25 in rt3_dn_b3 only (the centre tap's 0.140625 unchanged): 20 of the 54 tests fail, the
    reference comparisons from the first pass on (1x64: 0.11 there, 0.14-0.17 later);
  - ``sv += wt * cq.v`` for ``(wt * wt) * cq.v``: 19 fail, from the second pass on (1x64: 0.11 there, 0.20 later);
  - a reach of 1 in rt3_dn_tap_weight's call: 16 fail (1x64: 4.7e-3 at the first pass, 0.10 from the sixth).
tests/test_gpu_denoise.py cannot see any of them: kernels and restatement call the same header and change together."""
import ctypes as C

import numpy as np
import pytest

import denoise_lib as dl
import denoise_ref as ref
import oraclelib as ol
import path_aov_lib as pal
from rt3_b200 import abi, scenes

TAU = 2.0 ** -12
HULL_SLACK = 2.0 ** -18   # relative to the largest |e| of the footprint: a few float32 roundings of the weighted mean
ILL = 2.0 ** 12           # E[L^2] / var above which the float32 variance is held too inexact to compare with


def tau(sigma_normal=128.0):
    return TAU * max(1.0, sigma_normal / 128.0)


def rel_error(e32, e64):
    """max |e32 - e64| / max(|e64|, f), f = 10^-2 max |e64|; a non-finite value on either side counts as infinitely wrong."""
    e32 = np.asarray(e32, np.float64)
    f = 1e-2 * np.abs(e64[np.isfinite(e64)]).max(initial=0.0)
    with np.errstate(invalid="ignore", divide="ignore"):
        err = np.abs(e32 - e64) / np.maximum(np.abs(e64), f) if f > 0 else np.abs(e32 - e64)
    return float(np.nan_to_num(err, nan=np.inf).max())


def demodulated(rgb_out, albedo):
    """The filter's last demodulated colour from its remodulated float32 output (one more rounding: 2^-24 relative)."""
    return rgb_out.astype(np.float64) / np.maximum(albedo.astype(np.float64), ref.MIN_ALBEDO)


def restatement_passes(inp, flags=0, **dn):
    """The restatement's demodulated colour after every pass (one call per iteration count), and its last (frame, rgb)."""
    passes = []
    for i in range(1, dn.get("iterations", 5) + 1):
        frame, out = dl.oracle_denoise(*inp, flags=flags, **{**dn, "iterations": i})
        passes.append(demodulated(out, inp[1]))
    return passes, frame, out


def footprint(e, step, reach):
    """Per channel minimum and maximum of e over the taps at offsets step (dx, dy), |dx|, |dy| <= reach, inside the image."""
    h, w = e.shape[:2]
    taps = ref.Taps(h, w, reach * step)
    lo, hi = e.copy(), e.copy()
    for dy in range(-reach, reach + 1):
        for dx in range(-reach, reach + 1):
            q, ok = taps.view(e, dy * step, dx * step), taps.valid(dy * step, dx * step)[..., None]
            lo = np.where(ok, np.minimum(lo, q), lo)
            hi = np.where(ok, np.maximum(hi, q), hi)
    return lo, hi


def assert_in_hull(e_in, passes, what):
    """Each pass is a non-negative weighted mean of its 5x5 taps: per channel within their minimum and maximum."""
    for i, e_out in enumerate(passes):
        lo, hi = footprint(e_in, 2 ** i, 2)
        slack = HULL_SLACK * np.maximum(np.abs(lo), np.abs(hi))
        below, above = (lo - slack - e_out).max(), (e_out - hi - slack).max()
        assert np.isfinite(e_out).all() and below <= 0 and above <= 0, f"{what}: pass {i + 1} leaves its taps' hull by {max(below, above):.3g}"
        e_in = e_out


def frame_check(frame, res, albedo, tol, skip, gamma=True):
    """The 8-bit frame equals the reference's, except by 1 where the float64 level lies within the tolerance of a rounding
    boundary, and except on the pixels ``skip``. Returns (pixels off by one at a boundary, channels that break the rule)."""
    e64 = res["passes"][-1]
    d = np.maximum(albedo.astype(np.float64), ref.MIN_ALBEDO)
    de = tol * np.maximum(np.abs(e64), 1e-2 * np.abs(e64).max()) + 1e-6 * np.abs(e64)
    lo = np.floor(ref.resolve((e64 - de) * d, gamma)[0] + 0.5)
    hi = np.floor(ref.resolve((e64 + de) * d, gamma)[0] + 0.5)
    got, want = ol.unpack_rgb(frame), ol.unpack_rgb(res["frame"])
    near = (got != want) & (np.abs(got - want) == 1) & (got >= lo) & (got <= hi)
    bad = (got != want) & ~near & ~skip[..., None]
    return int(near.any(axis=-1).sum()), int(bad.sum())


# ---- inputs ----------------------------------------------------------------------------------------------------------------


def synthetic(h, w, seed=1, level=0.5, noise=0.3, miss=None, depth="flat", tilt=0.15, albedo=(0.2, 0.9)):
    """Radiance level (1 + noise u), u uniform in [-1, 1]; albedo uniform in ``albedo``; mean normals tilted up to ``tilt``
    radians from +z with lengths in [0.6, 1] (so w_n lies between 0 and 1); depth flat, a ramp or a step; misses (normal 0,
    depth +inf) in the left half, a ring or isolated pixels."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:h, :w].astype(np.float64)
    rgb = level * (1 + noise * rng.uniform(-1, 1, (h, w, 3)))
    alb = rng.uniform(*albedo, (h, w, 3))
    theta, phi = tilt * np.sqrt(rng.uniform(0, 1, (h, w))), rng.uniform(0, 2 * np.pi, (h, w))
    n = np.stack([np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)], -1) * rng.uniform(0.6, 1.0, (h, w, 1))
    z = {"flat": np.full((h, w), 2.0), "ramp": 1.0 + 0.04 * xx + 0.02 * yy, "step": np.where(xx < w / 2, 2.0, 5.0)}[depth]
    r = np.hypot(yy - (h - 1) / 2, xx - (w - 1) / 2)
    m = {None: np.zeros((h, w), bool), "half": xx < w // 2, "ring": (r > min(h, w) / 6) & (r < min(h, w) / 3),
         "isolated": rng.uniform(0, 1, (h, w)) < 0.04}[miss]
    n[m] = 0
    z[m] = np.inf
    return tuple(a.astype(np.float32) for a in (rgb, alb, n, z))


# id: (synthetic()'s arguments, the filter's parameters)  # worst error over the passes, measured
CASES = {
    "1x1": (dict(h=1, w=1), dict(iterations=8)),  # 0
    "1x64_isolated": (dict(h=1, w=64, miss="isolated", depth="ramp"), dict(iterations=8)),  # 4.2e-6
    "64x1_half": (dict(h=64, w=1, miss="half"), dict(iterations=5)),  # 3.8e-6
    "7x9_half": (dict(h=7, w=9, miss="half", depth="ramp"), dict(iterations=2)),  # 3.2e-6
    "31x8_ring": (dict(h=31, w=8, miss="ring", depth="step"), dict(iterations=5)),  # 4.5e-6
    "33x9_step": (dict(h=33, w=9, depth="step"), dict(iterations=8)),  # 4.3e-6
    "61x45_ring": (dict(h=61, w=45, miss="ring", depth="ramp"), dict(iterations=5)),  # 5.4e-6
    "61x45_isolated": (dict(h=61, w=45, miss="isolated", depth="step"), dict(iterations=8)),  # 5.8e-6
    "129x17_ramp": (dict(h=129, w=17, depth="ramp", tilt=0.3), dict(iterations=2)),  # 5.4e-6
    "17x129_half": (dict(h=17, w=129, miss="half", depth="ramp"), dict(iterations=1)),  # 5.7e-6
    "sigma_n_1": (dict(h=33, w=9, miss="ring", tilt=0.6), dict(iterations=5, sigma_normal=1.0)),  # 2.6e-7
    "sigma_n_7": (dict(h=61, w=45, depth="ramp", tilt=0.4), dict(iterations=5, sigma_normal=7.0)),  # 4.1e-7
    "sigma_n_1024": (dict(h=61, w=45, depth="ramp", tilt=0.04), dict(iterations=5, sigma_normal=1024.0)),  # 3.4e-5
    "sigma_l_1e-4": (dict(h=31, w=8, depth="ramp"), dict(iterations=5, sigma_luminance=1e-4)),  # 3.5e-6
    "sigma_l_1e4": (dict(h=31, w=8, depth="ramp"), dict(iterations=5, sigma_luminance=1e4)),  # 4.4e-6
    "sigma_z_1e-4": (dict(h=33, w=9, depth="ramp"), dict(iterations=5, sigma_depth=1e-4)),  # 2.0e-5
    "sigma_z_1e4": (dict(h=33, w=9, depth="step", miss="isolated"), dict(iterations=5, sigma_depth=1e4)),  # 1.0e-5
    "bright_dark_albedo": (dict(h=33, w=9, level=50.0, albedo=(0.0, 2e-3), miss="isolated"), dict(iterations=5)),  # 3.1e-6
}


def case_inputs(name):
    return synthetic(**CASES[name][0])


# ---- the primitives against libm ---------------------------------------------------------------------------------------------


def prim():
    lib = dl.oracle_lib()
    vp = C.c_void_p
    lib.orc_dn_exp_neg.argtypes = [vp, vp, C.c_size_t]
    lib.orc_dn_pow.argtypes = [vp, vp, vp, C.c_size_t]
    lib.orc_dn_make_guide.argtypes = [vp, vp, vp, C.c_size_t]
    return lib


def exp_neg(x):
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty_like(x)
    prim().orc_dn_exp_neg(x.ctypes.data, y.ctypes.data, x.size)
    return y


def exp_neg_error(x):
    """Relative error of rt3_dn_exp_neg against exp(-x) in float64; absolute where exp(-x) < 2^-126."""
    want = np.exp(-x.astype(np.float64))
    err = np.abs(exp_neg(x) - want)
    return np.where(want < 2.0 ** -126, err, err / want)


def test_exp_neg_against_libm():
    """Every 61st float32 in [0, 87) (18 million values): at most 4 units of 2^-24 relative. Measured: 9.7e-8 (1.6 units)."""
    x = np.arange(0, np.float32(87).view(np.uint32), 61, dtype=np.uint32).view(np.float32)
    worst = exp_neg_error(x).max()
    assert worst <= 4 * 2.0 ** -24, worst


def test_exp_neg_edges():
    """NaN, +inf and 87 give 0; 0 gives 1; the largest float32 below 87 and both sides of every k boundary (k +- 1/2) ln 2 are
    within the bound."""
    assert (exp_neg(np.array([np.nan, np.inf, 87.0, 88.0, 1e30])) == 0).all()
    assert exp_neg(np.zeros(1))[0] == 1.0
    k = np.arange(0, 126) + 0.5
    b = np.float32(k * np.log(2.0))
    x = np.concatenate([b, np.nextafter(b, np.float32(0)), np.nextafter(b, np.float32(np.inf)), [np.nextafter(np.float32(87), np.float32(0))]])
    assert exp_neg_error(x.astype(np.float32)).max() <= 4 * 2.0 ** -24


def test_pow_against_libm():
    """b^n for every n in 1..1024 over 4097 b in [0, 1] (a uniform grid and the 2048 float32 just below 1): at most n 2^-23
    relative (absolute 2^-126 where b^n is below 2^-126). Measured: 0.18 of the bound."""
    b = np.concatenate([np.linspace(0, 1, 2049), 1 - np.arange(1, 2049) * 2.0 ** -24]).astype(np.float32)
    n = np.arange(1, 1025, dtype=np.uint32)
    bb, nn = (np.ascontiguousarray(a) for a in np.broadcast_arrays(b[None, :], n[:, None]))
    y = np.empty(bb.shape, np.float32)
    prim().orc_dn_pow(bb.ctypes.data, nn.ctypes.data, y.ctypes.data, y.size)
    want = np.power(bb.astype(np.float64), nn.astype(np.float64))
    err = np.abs(y - want)
    ok = np.where(want < 2.0 ** -126, err <= 2.0 ** -126, err <= nn * 2.0 ** -23 * want)
    assert ok.all(), (bb[~ok][:5], nn[~ok][:5])


def make_guide(normal, depth):
    normal = np.ascontiguousarray(normal, np.float32)
    depth = np.ascontiguousarray(depth, np.float32)
    g = np.empty((depth.size, 4), np.float32)
    prim().orc_dn_make_guide(normal.ctypes.data, depth.ctypes.data, g.ctypes.data, depth.size)
    return g


@pytest.mark.parametrize("scale", [0.0, 1e-45, 1e-40, 1e-30, 1e-20, 1e-3, 1.0, 1e19, 1e20, 1e30, 3e38])
def test_guide_normalises_every_magnitude(scale):
    """n / |n| within 4 ulps (absolute 2^-126 for components that are not normal numbers), 0 where |n| = 0, depth passed on:
    for zero, denormal, tiny, huge and ordinary normals, including those whose squares under- or overflow float32."""
    rng = np.random.default_rng(5)
    n = rng.normal(size=(64, 3)) * np.float32(scale)
    n[:8, 1:] = 0                                  # a lone component: (s, 0, 0)
    n = n.astype(np.float32)
    z = np.float32(rng.uniform(0.5, 9, 64))
    z[::7] = np.inf
    g = make_guide(n, z)
    n64 = n.astype(np.float64)
    length = np.linalg.norm(n64, axis=-1, keepdims=True)
    want = n64 / np.where(length > 0, length, 1.0)
    assert np.array_equal(g[:, 3], z)
    bound = np.where(np.abs(want) < 2.0 ** -126, 2.0 ** -126, 4 * 2.0 ** -24 * np.abs(want))
    bad = (np.abs(g[:, :3] - want) > bound).any(axis=-1)
    assert not bad.any(), f"{bad.sum()} of 64 normals, e.g. {n[bad][0]} -> {g[bad][0, :3]}, want {want[bad][0]}"


# ---- the restatement against the reference -----------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def c1_inputs():
    """C1 at 200x113: the oracle path tracer's mean radiance at 16 spp (seed 1) and the 16-sample AOV restatement."""
    w, h = 200, 113
    scene, cam = scenes.rtiow_four_spheres(w, h)
    p = abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=16, max_depth=50, seed=1)
    _, acc, _ = ol.oracle_pathtrace(scene, cam, p, want_accum=True)
    rgb = (acc.astype(np.float64) / (16 * 16777216.0)).astype(np.float32)
    aov = pal.oracle_path_aovs(scene, cam, p)
    return rgb, aov["albedo"], aov["normal"], aov["hit_t"]


def ill_conditioned(res, iterations):
    """Per pass, the pixels whose result depends on an ill-conditioned luminance stop: where the 7x7 variance cancels by more
    than ILL (E[L^2] / var > ILL: float32 keeps fewer than 12 of its bits), and every pixel that later reads such a variance
    or a colour computed from one (the pass's 5x5 taps and g3x3's 3x3)."""
    h, w = res["cancellation"].shape
    tainted = ~(res["cancellation"] <= ILL)
    out = []
    for i in range(iterations):
        spread = tainted.copy()
        for step, reach in ((1, 1), (2 ** i, 2)):
            taps = ref.Taps(h, w, step * reach)
            for dy in range(-reach, reach + 1):
                for dx in range(-reach, reach + 1):
                    spread |= taps.view(tainted, dy * step, dx * step)
        tainted = spread
        out.append(tainted)
    return out


def compare(inp, passes, frame, what, flags=0, skip_ill=False, **dn):
    """Every pass of a filter's output (demodulated, from its float32 rgb) and its frame against the reference on the same
    inputs: the error per pass at most tau, every pass inside its taps' hull, the frame by the rounding-boundary rule. With
    ``skip_ill``, the pixels that depend on an ill-conditioned luminance stop (ill_conditioned()) are held to the hull only.
    Returns the worst error."""
    res = ref.denoise(*inp, gamma=not flags & abi.FLAG_NO_GAMMA, **dn)
    ill = ill_conditioned(res, len(passes)) if skip_ill else [np.zeros(inp[3].shape, bool)] * len(passes)
    errs = [rel_error(np.where(m[..., None], b, a), b) for a, b, m in zip(passes, res["passes"], ill)]
    t = tau(dn.get("sigma_normal", 128.0))
    assert max(errs) <= t, f"{what}: error per pass {['%.3g' % e for e in errs]} (tau {t:.3g})"
    assert_in_hull(res["input"], passes, what)
    near, bad = frame_check(frame, res, inp[1], t, ill[-1], gamma=not flags & abi.FLAG_NO_GAMMA)
    assert bad == 0, f"{what}: {bad} channels of the 8-bit frame differ from the reference's"
    print(f"{what}: worst error {max(errs):.3g} (tau {t:.3g}), {near} pixels off by one at an 8-bit rounding boundary"
          + (f", {ill[0].mean():.0%} to {ill[-1].mean():.0%} of the pixels ill-conditioned" if skip_ill else ""))
    return max(errs)


def check_against_reference(inp, what, flags=0, **dn):
    passes, frame, _ = restatement_passes(inp, flags=flags, **dn)
    return compare(inp, passes, frame, what, flags, **dn)


@pytest.mark.parametrize("name", list(CASES))
def test_synthetic_against_the_reference(name):
    check_against_reference(case_inputs(name), name, **CASES[name][1])


def test_no_gamma_against_the_reference():
    check_against_reference(case_inputs("61x45_ring"), "61x45_ring, no gamma", flags=abi.FLAG_NO_GAMMA, iterations=3)


@pytest.mark.parametrize("iterations", [1, 5, 8])
def test_c1_against_the_reference(c1_inputs, iterations):
    """Rendered radiance, misses, glass and metal: the worst error over the passes is measured at 9.1e-5 (1 iteration), 9.3e-5
    (5) and 9.3e-5 (8); two pixels of the 5- and 8-iteration frames are off by one at a rounding boundary."""
    check_against_reference(c1_inputs, f"C1 at {iterations} iterations", iterations=iterations)


def test_near_constant_stays_in_the_hull():
    """Noise 10^-6 of the level: the 7x7 variance E[L^2] - E[L]^2 has no correct digits in float32, so the luminance stop is
    ill-conditioned and the reference comparison does not apply; every pass still lies within its taps' hull."""
    inp = synthetic(33, 45, noise=1e-6, miss="ring", depth="ramp", seed=9)
    passes, _, _ = restatement_passes(inp, iterations=8)
    assert_in_hull(demodulated(inp[0], inp[1]), passes, "near constant")


def test_large_values_stay_in_the_hull():
    """Radiance 10^4 under albedo 0 (clamped to 10^-3): demodulated values of 10^7."""
    inp = synthetic(33, 45, level=1e4, albedo=(0.0, 1e-3), miss="isolated", depth="step", seed=4)
    passes, _, _ = restatement_passes(inp, iterations=8)
    assert_in_hull(demodulated(inp[0], inp[1]), passes, "large values")


# ---- every mutation of the reference is told apart -----------------------------------------------------------------------

# mutation: the case that tells it from the restatement by more than 10 tau = 2.4e-3  # the error measured there
KILLS = {
    "clamp_border": "33x9_step",           # 0.40
    "reach_one": "61x45_ring",             # 0.047
    "variance_w": "61x45_isolated",        # 0.34
    "g3x3_unweighted": "31x8_ring",        # 0.051
    "b3_flat": "61x45_ring",               # 0.40
    "no_centre_in_sum": "61x45_ring",      # inf (0 / 0 where no other tap has weight)
    "miss_depth_zero": "61x45_ring",       # 2.0
    "unnormalised_normals": "sigma_n_7",   # 2.0
    "step_linear": "61x45_isolated",       # 0.60
    "luminance_of_input": "61x45_ring",    # 0.29
}


def test_every_mutation_has_a_case():
    assert sorted(KILLS) == sorted(ref.MUTATIONS)
    assert set(KILLS.values()) <= set(CASES)


@pytest.mark.parametrize("mutation", list(ref.MUTATIONS))
def test_mutation_is_detected(mutation, request):
    name = KILLS[mutation]
    dn = CASES[name][1]
    inp = case_inputs(name)
    passes, _, _ = restatement_passes(inp, **dn)
    res = ref.denoise(*inp, mutation=mutation, **dn)
    err = max(rel_error(a, b) for a, b in zip(passes, res["passes"]))
    assert err > 10 * tau(dn.get("sigma_normal", 128.0)), f"{mutation} on {name}: {err:.3g}"
    print(f"{mutation} on {name}: {err:.3g}")


# ---- symmetries of the restatement ---------------------------------------------------------------------------------------


@pytest.mark.parametrize("name", ["61x45_ring", "129x17_ramp"])
def test_transpose_and_mirror(name):
    """Transposing all inputs transposes the output, mirroring them in x mirrors it: to within tau (the sums run in another
    order)."""
    inp = case_inputs(name)
    dn = CASES[name][1]
    _, base = dl.oracle_denoise(*inp, **dn)
    for what, f in (("transpose", lambda a: np.swapaxes(a, 0, 1)), ("mirror", lambda a: a[:, ::-1])):
        _, out = dl.oracle_denoise(*(np.ascontiguousarray(f(a)) for a in inp), **dn)
        err = rel_error(f(out), base.astype(np.float64))
        assert err <= TAU, f"{name} {what}: {err:.3g}"


@pytest.mark.parametrize("k", [-10, 3, 12])
def test_radiance_scale(k):
    """Radiance times 2^k gives the output times 2^k, to within tau rather than exactly: l_den's 1e-10 does not scale."""
    inp = case_inputs("61x45_isolated")
    _, base = dl.oracle_denoise(*inp, iterations=5)
    _, out = dl.oracle_denoise(inp[0] * np.float32(2.0 ** k), *inp[1:], iterations=5)
    err = rel_error(out.astype(np.float64) * 2.0 ** -k, base.astype(np.float64))
    assert err <= TAU, f"2^{k}: {err:.3g}"
