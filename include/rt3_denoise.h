/* rt3_denoise.h — per-pixel and per-tap arithmetic of the edge-avoiding à-trous denoiser (rt3_denoise, DESIGN.md 3.8).
 *
 * One definition for both sides: the kernels (csrc/rt3_denoise.cuh, nvcc -fmad=false) and the CPU restatement
 * (tests/denoise_oracle.c, gcc -ffp-contract=off) call these functions, so they agree bit for bit. As in rt3_rng.h,
 * every floating-point operation is one IEEE-754 binary32 operation in the order written; the only library call is
 * sqrtf (correctly rounded on both sides). exp(-x) is a fixed polynomial with range reduction, and the normal term's
 * power is taken by repeated squaring.
 *
 * Filter (Dammertz et al. 2010; the spatial filter of SVGF, Schied et al. 2017, without its temporal part):
 *   e = c / max(a, 1e-3) per channel (demodulated radiance), L(e) = 0.2126 r + 0.7152 g + 0.0722 b;
 *   guide = (normalised mean normal n^, 0 where |n| = 0; depth z, +inf on a miss);
 *   variance: over 7x7, weights w_z w_n (reach 1 per pixel of offset), max(0, E[L^2] - E[L]^2);
 *   pass i (step s = 2^i), 5x5 taps at offsets s (dx, dy), B3-spline h = (1/16, 1/4, 3/8, 1/4, 1/16):
 *     w = ((h_y h_x) w_n) exp(-(x_z + x_l)),
 *     x_z = |z_p - z_q| / ((sigma_z z_p) (s max(|dx|, |dy|)) + 1e-6)   (w_z = exp(-x_z)),
 *     x_l = |L_p - L_q| / (sigma_l sqrt(g3x3(var)_p) + 1e-10)           (w_l = exp(-x_l)),
 *     w_n = max(0, n^_p . n^_q)^sigma_n;
 *     two misses: x_z = 0, w_n = 1; a miss and a hit: w = 0; the centre tap: w = h_2 h_2 = 9/64;
 *     out = (e_p + sum w (e_q - e_p) / sum w, sum w^2 var_q / (sum w)^2): the weighted mean, written as the centre plus
 *     the weighted mean of the differences so that a constant image comes back exactly; taps outside the image are skipped;
 *   g3x3(var)_p: 3x3 taps at step 1 with weights (g_y g_x) w_z w_n, g = (1/4, 1/2, 1/4), normalised.
 * Sums run rows -r..r outer, columns -r..r inner. */
#ifndef RT3_DENOISE_H
#define RT3_DENOISE_H

#include <stdint.h>
#include <string.h>

#include "rt3_rng.h" /* RT3_HD */
#include "rt3cuda.h"  /* rt3_denoise_params */

#define RT3_DN_MIN_ALBEDO 1e-3f
#define RT3_DN_EPS_Z 1e-6f
#define RT3_DN_EPS_L 1e-10f
#define RT3_DN_MAX_ITERATIONS 8u
#define RT3_DN_MAX_NORMAL_POWER 1024.0f
#define RT3_DN_FLT_MAX 3.402823466e38f

#if defined(__CUDACC__)
#define RT3_DN_ALIGN16 __align__(16)
#define RT3_DN_RESTRICT __restrict__
#define RT3_DN_UNROLL _Pragma("unroll")
#else
#define RT3_DN_ALIGN16 __attribute__((aligned(16)))
#define RT3_DN_RESTRICT restrict
#define RT3_DN_UNROLL
#endif

/* Per-pixel guide: normalised normal and depth. */
typedef struct RT3_DN_ALIGN16 rt3_dn_guide {
    float nx, ny, nz, z;
} rt3_dn_guide;

/* Per-pixel filter state: demodulated colour and the variance of its luminance (before the passes: the luminance). */
typedef struct RT3_DN_ALIGN16 rt3_dn_px {
    float r, g, b, v;
} rt3_dn_px;

/* exp(-x) for x >= 0 (NaN and x >= 87 give 0). x = k ln2 + r with k = (int) (x log2(e) + 1/2) and |r| <= ln2 / 2 (Cody-Waite:
 * ln2 = 0.693359375 - 2.12194440e-4, the first part exact in 9 bits so k * it is exact); exp(-r) by its Taylor polynomial of
 * degree 7 in Horner form (truncation error below 5e-9 relative); 2^-k from the exponent bits (k <= 126: a normal number). */
RT3_HD float rt3_dn_exp_neg(float x) {
    if (!(x < 87.0f)) { return 0.0f; }
    const int k = (int) (x * 1.44269504f + 0.5f);
    const float kf = (float) k;
    const float t = -((x - kf * 0.693359375f) + kf * 2.12194440e-4f);
    float p = 1.984126984e-4f;          /* 1/5040 */
    p = 1.388888889e-3f + t * p;        /* 1/720 */
    p = 8.333333333e-3f + t * p;        /* 1/120 */
    p = 4.166666667e-2f + t * p;        /* 1/24 */
    p = 1.666666667e-1f + t * p;        /* 1/6 */
    p = 0.5f + t * p;
    p = 1.0f + t * p;
    p = 1.0f + t * p;
    const uint32_t bits = (uint32_t) (127 - k) << 23;
    float scale;
#if defined(__CUDA_ARCH__)
    scale = __uint_as_float(bits);
#else
    memcpy(&scale, &bits, sizeof scale);
#endif
    return p * scale;
}

/* b^n by repeated squaring, lowest bit first. */
RT3_HD float rt3_dn_pow(float b, uint32_t n) {
    float r = 1.0f;
    while (n) {
        if (n & 1u) { r = r * b; }
        n >>= 1;
        if (n) { b = b * b; }
    }
    return r;
}

RT3_HD float rt3_dn_luminance(float r, float g, float b) { return (0.2126f * r + 0.7152f * g) + 0.0722f * b; }

/* max(a, 1e-3): the albedo the radiance is divided by (demodulation) and multiplied by again after the last pass. */
RT3_HD float rt3_dn_albedo(float a) { return a > RT3_DN_MIN_ALBEDO ? a : RT3_DN_MIN_ALBEDO; }

/* n / |n|, 0 where |n| = 0. Where |n|^2 would leave the normal range (|n| below about 2^-50 or above 2^50), n is first scaled
 * by 2^100 or 2^-100: exact, so the direction is kept, and no other normal takes this branch or changes a bit. */
RT3_HD rt3_dn_guide rt3_dn_make_guide(float nx, float ny, float nz, float hit_t) {
    rt3_dn_guide g;
    float len2 = (nx * nx + ny * ny) + nz * nz;
    if (len2 < 0x1p-100f || len2 > 0x1p100f) {
        const float s = len2 < 0x1p-100f ? 0x1p100f : 0x1p-100f;
        nx = nx * s; ny = ny * s; nz = nz * s;
        len2 = (nx * nx + ny * ny) + nz * nz;
    }
    if (len2 > 0.0f) {
        const float inv = 1.0f / sqrtf(len2);
        g.nx = nx * inv; g.ny = ny * inv; g.nz = nz * inv;
    } else {
        g.nx = 0.0f; g.ny = 0.0f; g.nz = 0.0f;
    }
    g.z = hit_t;
    return g;
}

/* Geometry terms of tap q seen from p at `reach` pixels (s max(|dx|, |dy|)): returns w_n and writes x_z; returns -1 when
 * exactly one of the two is a miss (the tap's weight is 0). */
RT3_HD float rt3_dn_geometry(rt3_dn_guide p, rt3_dn_guide q, float sigma_z, uint32_t reach, uint32_t n_pow, float* x_z) {
    const int miss_p = p.z > RT3_DN_FLT_MAX, miss_q = q.z > RT3_DN_FLT_MAX;
    *x_z = 0.0f;
    if (miss_p != miss_q) { return -1.0f; }
    if (miss_p) { return 1.0f; }
    const float dz = p.z - q.z;
    *x_z = (dz < 0.0f ? -dz : dz) / ((sigma_z * p.z) * (float) reach + RT3_DN_EPS_Z);
    const float c = (p.nx * q.nx + p.ny * q.ny) + p.nz * q.nz;
    return rt3_dn_pow(c > 0.0f ? c : 0.0f, n_pow);
}

/* w_z w_n: the weight of a variance tap (the 7x7 estimate and g3x3), without its spatial factor. */
RT3_HD float rt3_dn_geometry_weight(rt3_dn_guide p, rt3_dn_guide q, float sigma_z, uint32_t reach, uint32_t n_pow) {
    float x_z;
    const float w_n = rt3_dn_geometry(p, q, sigma_z, reach, n_pow, &x_z);
    if (w_n < 0.0f) { return 0.0f; }
    return w_n * rt3_dn_exp_neg(x_z);
}

/* Full à-trous tap weight ((h_y h_x) w_n) exp(-(x_z + x_l)), l_den = sigma_l sqrt(g3x3(var)_p) + 1e-10. */
RT3_HD float rt3_dn_tap_weight(float hyx, rt3_dn_guide p, rt3_dn_guide q, float l_p, float l_q, float l_den, float sigma_z, uint32_t reach,
                               uint32_t n_pow) {
    float x_z;
    const float w_n = rt3_dn_geometry(p, q, sigma_z, reach, n_pow, &x_z);
    if (w_n < 0.0f) { return 0.0f; }
    const float dl = l_p - l_q;
    const float x_l = (dl < 0.0f ? -dl : dl) / l_den;
    return (hyx * w_n) * rt3_dn_exp_neg(x_z + x_l);
}

RT3_HD float rt3_dn_b3(int i) { return i == 0 ? 0.375f : (i == 1 || i == -1) ? 0.25f : 0.0625f; }
RT3_HD float rt3_dn_g3(int i) { return i == 0 ? 0.5f : 0.25f; }

RT3_HD int rt3_dn_max_abs(int a, int b) { a = a < 0 ? -a : a; b = b < 0 ? -b : b; return a < b ? b : a; }

/* Prepare: demodulated colour with its luminance in v, and the guide, from radiance c, albedo a, normal n and depth t. */
RT3_HD void rt3_dn_prepare_px(const float* c, const float* a, const float* n, float t, rt3_dn_px* px, rt3_dn_guide* guide) {
    px->r = c[0] / rt3_dn_albedo(a[0]);
    px->g = c[1] / rt3_dn_albedo(a[1]);
    px->b = c[2] / rt3_dn_albedo(a[2]);
    px->v = rt3_dn_luminance(px->r, px->g, px->b);
    *guide = rt3_dn_make_guide(n[0], n[1], n[2], t);
}

/* Variance of the luminance at (x, y) from the prepared state (v = L): 7x7, weights w_z w_n, the centre 1. */
RT3_HD float rt3_dn_variance_px(const rt3_dn_px* RT3_DN_RESTRICT col, const rt3_dn_guide* RT3_DN_RESTRICT guide, uint32_t w, uint32_t h, uint32_t x,
                                uint32_t y, float sigma_z, uint32_t n_pow) {
    const rt3_dn_guide gp = guide[(size_t) y * w + x];
    float sw = 0.0f, m1 = 0.0f, m2 = 0.0f;
    RT3_DN_UNROLL
    for (int dy = -3; dy <= 3; dy++) {
        const int qy = (int) y + dy;
        if (qy < 0 || qy >= (int) h) { continue; }
        RT3_DN_UNROLL
        for (int dx = -3; dx <= 3; dx++) {
            const int qx = (int) x + dx;
            if (qx < 0 || qx >= (int) w) { continue; }
            const size_t q = (size_t) qy * w + (size_t) qx;
            const float l = col[q].v;
            const float wt = (dx == 0 && dy == 0) ? 1.0f : rt3_dn_geometry_weight(gp, guide[q], sigma_z, (uint32_t) rt3_dn_max_abs(dx, dy), n_pow);
            sw = sw + wt;
            m1 = m1 + wt * l;
            m2 = m2 + (wt * l) * l;
        }
    }
    const float mean = m1 / sw;
    const float var = m2 / sw - mean * mean;
    return var > 0.0f ? var : 0.0f;
}

/* One à-trous pass at (x, y) with step `step`. */
RT3_HD rt3_dn_px rt3_dn_atrous_px(const rt3_dn_px* RT3_DN_RESTRICT col, const rt3_dn_guide* RT3_DN_RESTRICT guide, uint32_t w, uint32_t h, uint32_t x,
                                  uint32_t y, uint32_t step, float sigma_l, float sigma_z, uint32_t n_pow) {
    const size_t p = (size_t) y * w + x;
    const rt3_dn_px cp = col[p];
    const rt3_dn_guide gp = guide[p];
    /* g3x3(var)_p */
    float gs = 0.0f, gv = 0.0f;
    RT3_DN_UNROLL
    for (int dy = -1; dy <= 1; dy++) {
        const int qy = (int) y + dy;
        if (qy < 0 || qy >= (int) h) { continue; }
        RT3_DN_UNROLL
        for (int dx = -1; dx <= 1; dx++) {
            const int qx = (int) x + dx;
            if (qx < 0 || qx >= (int) w) { continue; }
            const size_t q = (size_t) qy * w + (size_t) qx;
            const float wt = (dx == 0 && dy == 0) ? 0.25f : (rt3_dn_g3(dy) * rt3_dn_g3(dx)) * rt3_dn_geometry_weight(gp, guide[q], sigma_z, 1u, n_pow);
            gs = gs + wt;
            gv = gv + wt * col[q].v;
        }
    }
    const float l_den = sigma_l * sqrtf(gv / gs) + RT3_DN_EPS_L;
    const float l_p = rt3_dn_luminance(cp.r, cp.g, cp.b);
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
    RT3_DN_UNROLL
    for (int dy = -2; dy <= 2; dy++) {
        const int qy = (int) y + dy * (int) step;
        if (qy < 0 || qy >= (int) h) { continue; }
        RT3_DN_UNROLL
        for (int dx = -2; dx <= 2; dx++) {
            const int qx = (int) x + dx * (int) step;
            if (qx < 0 || qx >= (int) w) { continue; }
            const size_t q = (size_t) qy * w + (size_t) qx;
            const rt3_dn_px cq = col[q];
            const float wt = (dx == 0 && dy == 0) ? 0.140625f /* (3/8)^2 */
                : rt3_dn_tap_weight(rt3_dn_b3(dy) * rt3_dn_b3(dx), gp, guide[q], l_p, rt3_dn_luminance(cq.r, cq.g, cq.b), l_den, sigma_z,
                                    step * (uint32_t) rt3_dn_max_abs(dx, dy), n_pow);
            sw = sw + wt;
            sr = sr + wt * (cq.r - cp.r);
            sg = sg + wt * (cq.g - cp.g);
            sb = sb + wt * (cq.b - cp.b);
            sv = sv + (wt * wt) * cq.v;
        }
    }
    rt3_dn_px out;
    out.r = cp.r + sr / sw; out.g = cp.g + sg / sw; out.b = cp.b + sb / sw;
    out.v = sv / (sw * sw);
    return out;
}

/* After the last pass: the filtered colour times max(a, 1e-3) again. */
RT3_HD float rt3_dn_remodulate(float e, float a) { return e * rt3_dn_albedo(a); }

/* NULL when the parameters are valid, else what is wrong with them. sigma_normal is the integer exponent of the normal term. */
static inline const char* rt3_dn_check_params(const rt3_denoise_params* p) {
    if (!p) { return "params is NULL"; }
    if (p->iterations < 1 || p->iterations > RT3_DN_MAX_ITERATIONS) { return "iterations must be in 1..8"; }
    if (!(p->sigma_luminance > 0.0f && p->sigma_luminance <= RT3_DN_FLT_MAX)) { return "sigma_luminance must be finite and > 0"; }
    if (!(p->sigma_depth > 0.0f && p->sigma_depth <= RT3_DN_FLT_MAX)) { return "sigma_depth must be finite and > 0"; }
    if (!(p->sigma_normal >= 1.0f && p->sigma_normal <= RT3_DN_MAX_NORMAL_POWER) || (float) (uint32_t) p->sigma_normal != p->sigma_normal) {
        return "sigma_normal must be a whole number in 1..1024 (the exponent of the normal term)";
    }
    return NULL;
}

#endif /* RT3_DENOISE_H */
