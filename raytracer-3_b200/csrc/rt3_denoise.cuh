/* rt3_denoise.cuh — kernels of rt3_denoise (DESIGN.md 3.8): the edge-avoiding à-trous filter on the radiance of the last
 * path-traced render, guided by the last path-traced AOVs. The arithmetic is include/rt3_denoise.h's; these kernels only
 * load, call it and store. Every kernel but the stage covers the whole frame (rt3_denoise needs part_count <= 1), one
 * thread per pixel.
 *
 *   denoise_prepare_kernel   : radiance (mean_radiance) / albedo -> colour + luminance, normal + depth -> guide.
 *   denoise_stage_kernel     : the same for a partition's owned rows, into a stage buffer (rt3_denoise_stage), + row fingerprints.
 *   denoise_variance_kernel  : 7x7 luminance variance.
 *   denoise_atrous_kernel<F> : one 5x5 pass at step 2^i; F = the last pass, which remodulates and resolves like resolve_kernel.
 *   denoise_temporal_kernel  : rt3_denoise_temporal: prepare, reproject into the previous camera, accumulate the history.
 *   denoise_temporal_variance_kernel : its variance, from the luminance moments or the 7x7 estimate.
 *
 * Taps are read straight from global memory through L1 (float4 loads): a 2^i-strided 5x5 footprint is 25 float4 of colour
 * and 25 of guide, all but the far ones shared with the neighbouring threads of the CTA. */
#pragma once

#include "rt3_denoise.h"
#include "rt3_device.cuh"
#include "rt3_kernels.cuh" /* owned_row_to_global, mean_radiance */

#define RT3_DN_BLOCK_X 32
#define RT3_DN_BLOCK_Y 8

/* Loads pixel idx of the render (its mean radiance) and of its albedo, normal and depth AOVs and prepares it
 * (rt3_dn_prepare_px). Returns the depth; the albedo is returned in a[], for the stage kernel to store. */
__device__ __forceinline__ float dn_load_prepare(const rt3_kparams& P, const unsigned long long* __restrict__ accum, const float* __restrict__ albedo,
                                                 const float* __restrict__ normal, const float* __restrict__ depth, size_t idx, float a[3], rt3_dn_px* px,
                                                 rt3_dn_guide* g) {
    float c[3], n[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        c[k] = mean_radiance(P, accum, idx, k);
        a[k] = albedo[3 * idx + k];
        n[k] = normal[3 * idx + k];
    }
    const float z = depth[idx];
    rt3_dn_prepare_px(c, a, n, z, px, g);
    return z;
}

__global__ void __launch_bounds__(256) denoise_prepare_kernel(rt3_kparams P, const unsigned long long* __restrict__ accum, const float* __restrict__ albedo,
                                                             const float* __restrict__ normal, const float* __restrict__ depth, rt3_dn_px* __restrict__ col,
                                                             rt3_dn_guide* __restrict__ guide) {
    const unsigned long long idx = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P.n_pixels) { return; }
    float a[3];
    rt3_dn_px px;
    rt3_dn_guide g;
    dn_load_prepare(P, accum, albedo, normal, depth, idx, a, &px, &g);
    col[idx] = px;
    guide[idx] = g;
}

/* rt3_denoise_stage: denoise_prepare_kernel's step for the rows a partitioned render owns (one thread per owned pixel, the
 * row mapping of resolve_kernel), stored at full-frame indices into the stage's colour, guide and albedo planes, which may
 * live on another GPU; the first thread of each row also stores the row's fingerprint. */
__global__ void __launch_bounds__(256) denoise_stage_kernel(rt3_kparams P, const unsigned long long* __restrict__ accum, const float* __restrict__ albedo,
                                                           const float* __restrict__ normal, const float* __restrict__ depth, rt3_dn_px* __restrict__ col,
                                                           rt3_dn_guide* __restrict__ guide, float* __restrict__ stage_albedo,
                                                           unsigned long long* __restrict__ row_fingerprint, unsigned long long fingerprint) {
    const unsigned long long p = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pixels) { return; }
    const uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    const uint32_t y = owned_row_to_global(P, local_row);
    const size_t idx = (size_t) y * P.width + x;
    float a[3];
    rt3_dn_px px;
    rt3_dn_guide g;
    dn_load_prepare(P, accum, albedo, normal, depth, idx, a, &px, &g);
    col[idx] = px;
    guide[idx] = g;
#pragma unroll
    for (int k = 0; k < 3; k++) { stage_albedo[3 * idx + k] = a[k]; }
    if (x == 0) { row_fingerprint[y] = fingerprint; }
}

__global__ void __launch_bounds__(RT3_DN_BLOCK_X * RT3_DN_BLOCK_Y) denoise_variance_kernel(uint32_t w, uint32_t h, float sigma_z, uint32_t n_pow,
                                                                                         const rt3_dn_px* __restrict__ col, const rt3_dn_guide* __restrict__ guide,
                                                                                         rt3_dn_px* __restrict__ out) {
    const uint32_t x = blockIdx.x * RT3_DN_BLOCK_X + threadIdx.x, y = blockIdx.y * RT3_DN_BLOCK_Y + threadIdx.y;
    if (x >= w || y >= h) { return; }
    const size_t p = (size_t) y * w + x;
    rt3_dn_px px = col[p];
    px.v = rt3_dn_variance_px(col, guide, w, h, x, y, sigma_z, n_pow);
    out[p] = px;
}

template <bool FINAL>
__global__ void __launch_bounds__(RT3_DN_BLOCK_X * RT3_DN_BLOCK_Y) denoise_atrous_kernel(uint32_t w, uint32_t h, uint32_t step, float sigma_l, float sigma_z,
                                                                                       uint32_t n_pow, const rt3_dn_px* __restrict__ col,
                                                                                       const rt3_dn_guide* __restrict__ guide, rt3_dn_px* __restrict__ out,
                                                                                       const float* __restrict__ albedo, bool gamma, uint32_t* __restrict__ frame,
                                                                                       float* __restrict__ rgb) {
    const uint32_t x = blockIdx.x * RT3_DN_BLOCK_X + threadIdx.x, y = blockIdx.y * RT3_DN_BLOCK_Y + threadIdx.y;
    if (x >= w || y >= h) { return; }
    const size_t p = (size_t) y * w + x;
    const rt3_dn_px f = rt3_dn_atrous_px(col, guide, w, h, x, y, step, sigma_l, sigma_z, n_pow);
    if (!FINAL) {
        out[p] = f;
        return;
    }
    const float r = rt3_dn_remodulate(f.r, albedo[3 * p]), g = rt3_dn_remodulate(f.g, albedo[3 * p + 1]), b = rt3_dn_remodulate(f.b, albedo[3 * p + 2]);
    if (rgb) { rgb[3 * p] = r; rgb[3 * p + 1] = g; rgb[3 * p + 2] = b; }
    frame[p] = gamma ? (unorm8(sqrtf(r)) << 24) | (unorm8(sqrtf(g)) << 16) | (unorm8(sqrtf(b)) << 8) | 0xFFu
                     : (unorm8(r) << 24) | (unorm8(g) << 16) | (unorm8(b) << 8) | 0xFFu;
}

/* rt3_denoise_temporal, steps 1-6 (include/rt3_denoise.h): prepares pixel p as denoise_prepare_kernel does (the render's
 * kparams P), regenerates the primary ray of sample first_sample of the AOV call (kparams A, start_path), reprojects its
 * surface point into the previous camera and accumulates the previous history (read only when `have_prev`) into the next
 * one. Writes the accumulated colour (v = its luminance) and the guide for the variance and à-trous passes, and the
 * history length to `length` when it is not null. */
__global__ void __launch_bounds__(RT3_DN_BLOCK_X * RT3_DN_BLOCK_Y) denoise_temporal_kernel(
    rt3_kparams P, rt3_kparams A, rt3_camera cur_cam, rt3_camera prev_cam, rt3_denoise_temporal_params tp, bool have_prev,
    const unsigned long long* __restrict__ accum, const float* __restrict__ albedo, const float* __restrict__ normal, const float* __restrict__ depth,
    const rt3_dn_hist* __restrict__ prev_col, const rt3_dn_moments* __restrict__ prev_mom, const rt3_dn_guide* __restrict__ prev_guide,
    rt3_dn_hist* __restrict__ next_col, rt3_dn_moments* __restrict__ next_mom, rt3_dn_guide* __restrict__ next_guide, rt3_dn_px* __restrict__ col,
    rt3_dn_guide* __restrict__ guide, float* __restrict__ length) {
    const uint32_t w = P.width, h = P.height;
    const uint32_t x = blockIdx.x * RT3_DN_BLOCK_X + threadIdx.x, y = blockIdx.y * RT3_DN_BLOCK_Y + threadIdx.y;
    if (x >= w || y >= h) { return; }
    const size_t idx = (size_t) y * w + x;
    float a[3];
    rt3_dn_px e;
    rt3_dn_guide g;
    const float z = dn_load_prepare(P, accum, albedo, normal, depth, idx, a, &e, &g);
    int have = 0;
    float px = 0.0f, py = 0.0f, dist = 0.0f;
    if (have_prev) {
        rt3_cam_view C;
        C.origin = v3(cur_cam.origin[0], cur_cam.origin[1], cur_cam.origin[2]);
        C.hor = v3(cur_cam.horizontal[0], cur_cam.horizontal[1], cur_cam.horizontal[2]);
        C.ver = v3(cur_cam.vertical[0], cur_cam.vertical[1], cur_cam.vertical[2]);
        C.llc = v3(cur_cam.lower_left_corner[0], cur_cam.lower_left_corner[1], cur_cam.lower_left_corner[2]);
        C.lens_u = v3(cur_cam.lens_u[0], cur_cam.lens_u[1], cur_cam.lens_u[2]);
        C.lens_v = v3(cur_cam.lens_v[0], cur_cam.lens_v[1], cur_cam.lens_v[2]);
        C.lens_radius = cur_cam.lens_radius;
        C.wm1 = (float) A.width - 1.0f; C.hm1 = (float) A.height - 1.0f;
        rt3_path s;
        start_path(s, C, A, (uint32_t) idx, 0u); /* the AOVs cover the whole frame: compact index = pixel index */
        have = rt3_dn_reproject(cur_cam, prev_cam, w, h, x, y, s.o.x, s.o.y, s.o.z, s.d.x, s.d.y, s.d.z, z, &px, &py, &dist);
    }
    rt3_dn_hist hc;
    rt3_dn_moments hm;
    rt3_dn_accumulate_px(prev_col, prev_mom, prev_guide, w, h, have, px, py, dist, e, g, &tp, &hc, &hm);
    next_col[idx] = hc;
    next_mom[idx] = hm;
    next_guide[idx] = g;
    rt3_dn_px acc;
    acc.r = hc.r; acc.g = hc.g; acc.b = hc.b;
    acc.v = rt3_dn_luminance(hc.r, hc.g, hc.b);
    col[idx] = acc;
    guide[idx] = g;
    if (length) { length[idx] = hc.n; }
}

/* rt3_denoise_temporal, step 7: the accumulated colour with its luminance variance (from the moments from 4 frames on,
 * else denoise_variance_kernel's 7x7 estimate) into `out`, the input of the à-trous passes. */
__global__ void __launch_bounds__(RT3_DN_BLOCK_X * RT3_DN_BLOCK_Y) denoise_temporal_variance_kernel(uint32_t w, uint32_t h, float sigma_z, uint32_t n_pow,
                                                                                                  const rt3_dn_px* __restrict__ col, const rt3_dn_guide* __restrict__ guide,
                                                                                                  const rt3_dn_hist* __restrict__ hist, const rt3_dn_moments* __restrict__ mom,
                                                                                                  rt3_dn_px* __restrict__ out) {
    const uint32_t x = blockIdx.x * RT3_DN_BLOCK_X + threadIdx.x, y = blockIdx.y * RT3_DN_BLOCK_Y + threadIdx.y;
    if (x >= w || y >= h) { return; }
    const size_t p = (size_t) y * w + x;
    rt3_dn_px px = col[p];
    px.v = rt3_dn_temporal_variance_px(col, guide, hist[p].n, mom[p], w, h, x, y, sigma_z, n_pow);
    out[p] = px;
}
