/* denoise_oracle.c — CPU restatement of rt3_denoise and rt3_denoise_temporal (TEST INFRASTRUCTURE, plain C11, built by
 * tests/denoise_lib.py with the oracle's flags: -O2 -ffp-contract=off -fno-fast-math).
 *
 * The filter's and the temporal arithmetic are include/rt3_denoise.h, the same functions the kernels call; this file
 * restates only what the kernels do around them: the order of the passes, the ping-pong buffers and the resolve
 * (resolve_kernel's gamma, unorm8 and packing; the oracle's unorm8 is the kernels'). Its inputs are the arrays
 * rt3_read_radiance and rt3_render_path_aovs return, so it can be fed the GPU's own inputs, or synthetic ones. The rays
 * rt3_denoise_temporal reprojects are primary_ray's of the AOV restatement (tests/path_aov_oracle.c), compiled into this
 * unit with the oracle it includes (for_each_row, unorm8). Any width and height >= 1 are accepted (the library renders
 * nothing under 2x2). */
#include "path_aov_oracle.c"
#include "rt3_denoise.h"

int orc_denoise(uint32_t w, uint32_t h, const float* rgb, const float* albedo, const float* normal, const float* depth, const rt3_denoise_params* p,
                uint32_t flags, uint32_t* frame, float* rgb_out, int n_threads);
const char* orc_denoise_check(const rt3_denoise_params* p);
void orc_dn_exp_neg(const float* x, float* y, size_t count);
void orc_dn_pow(const float* b, const uint32_t* n_pow, float* y, size_t count);
void orc_dn_make_guide(const float* normal, const float* depth, float* guide, size_t count);
int orc_denoise_temporal(uint32_t w, uint32_t h, const float* rgb, const float* albedo, const float* normal, const float* depth, const rt3_camera* cam,
                         const rt3_params* aov, const rt3_camera* prev_cam, int have_prev, const rt3_dn_hist* prev_col, const rt3_dn_moments* prev_mom,
                         const rt3_dn_guide* prev_guide, const rt3_denoise_temporal_params* tp, uint32_t flags, rt3_dn_hist* next_col,
                         rt3_dn_moments* next_mom, rt3_dn_guide* next_guide, uint32_t* frame, float* rgb_out, float* length, int n_threads);
const char* orc_denoise_temporal_check(const rt3_denoise_temporal_params* p);
int orc_dn_reproject(const rt3_camera* cur, const rt3_camera* prev, uint32_t w, uint32_t h, const float* xy, const float* ray, const float* depth,
                     float* pos, size_t count);
void orc_dn_primary_rays(const rt3_camera* cam, const rt3_params* aov, float* rays);

typedef struct {
    uint32_t w, h, step, n_pow, final_pass, gamma;
    float sigma_l, sigma_z;
    const float *rgb, *albedo, *normal, *depth;
    rt3_dn_px *in, *out;
    rt3_dn_guide* guide;
    uint32_t* frame;
    float* rgb_out;
    /* rt3_denoise_temporal's only */
    const rt3_camera *cam, *prev_cam;
    const rt3_params* aov;
    int have_prev;
    const rt3_dn_hist* prev_col;
    const rt3_dn_moments* prev_mom;
    const rt3_dn_guide* prev_guide;
    const rt3_denoise_temporal_params* tp;
    rt3_dn_hist* next_col;
    rt3_dn_moments* next_mom;
    rt3_dn_guide* next_guide;
    float* length;
} dn_job;

typedef void (*dn_row)(void* ctx, uint32_t y);

/* denoise_prepare_kernel */
static void prepare_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        rt3_dn_prepare_px(j->rgb + 3 * i, j->albedo + 3 * i, j->normal + 3 * i, j->depth[i], &j->out[i], &j->guide[i]);
    }
}

/* denoise_variance_kernel */
static void variance_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        j->out[i] = j->in[i];
        j->out[i].v = rt3_dn_variance_px(j->in, j->guide, j->w, j->h, x, y, j->sigma_z, j->n_pow);
    }
}

/* denoise_temporal_kernel: prepare, primary ray of sample first_sample of the AOV call, reprojection, accumulation. */
static void temporal_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        rt3_dn_px e;
        rt3_dn_guide g;
        rt3_dn_prepare_px(j->rgb + 3 * i, j->albedo + 3 * i, j->normal + 3 * i, j->depth[i], &e, &g);
        int have = 0;
        float px = 0.0f, py = 0.0f, dist = 0.0f;
        if (j->have_prev) {
            v3 o, d = primary_ray(j->cam, j->aov, x, y, j->aov->first_sample, &o);
            have = rt3_dn_reproject(*j->cam, *j->prev_cam, j->w, j->h, x, y, o.x, o.y, o.z, d.x, d.y, d.z, j->depth[i], &px, &py, &dist);
        }
        rt3_dn_hist hc;
        rt3_dn_moments hm;
        rt3_dn_accumulate_px(j->prev_col, j->prev_mom, j->prev_guide, j->w, j->h, have, px, py, dist, e, g, j->tp, &hc, &hm);
        j->next_col[i] = hc;
        j->next_mom[i] = hm;
        j->next_guide[i] = g;
        j->out[i].r = hc.r; j->out[i].g = hc.g; j->out[i].b = hc.b;
        j->out[i].v = rt3_dn_luminance(hc.r, hc.g, hc.b);
        j->guide[i] = g;
        if (j->length) { j->length[i] = hc.n; }
    }
}

/* denoise_temporal_variance_kernel */
static void temporal_variance_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        j->out[i] = j->in[i];
        j->out[i].v = rt3_dn_temporal_variance_px(j->in, j->guide, j->next_col[i].n, j->next_mom[i], j->w, j->h, x, y, j->sigma_z, j->n_pow);
    }
}

/* denoise_atrous_kernel: one pass, the last one remodulating and resolving like resolve_kernel. */
static void atrous_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        const rt3_dn_px f = rt3_dn_atrous_px(j->in, j->guide, j->w, j->h, x, y, j->step, j->sigma_l, j->sigma_z, j->n_pow);
        if (!j->final_pass) { j->out[i] = f; continue; }
        const float e[3] = { f.r, f.g, f.b };
        uint32_t ch[3];
        for (int k = 0; k < 3; k++) {
            const float m = rt3_dn_remodulate(e[k], j->albedo[3 * i + k]);
            if (j->rgb_out) { j->rgb_out[3 * i + k] = m; }
            ch[k] = unorm8(j->gamma ? sqrtf(m) : m);
        }
        if (j->frame) { j->frame[i] = (ch[0] << 24) | (ch[1] << 16) | (ch[2] << 8) | 0xFFu; }
    }
}

/* The passes of both calls over the job's inputs: `prepare` into col[1] and the guides, `variance` into col[0], then the
 * `iterations` à-trous passes ping-ponging through col. */
static int run_passes(dn_job* j, const rt3_denoise_params* p, uint32_t flags, dn_row prepare, dn_row variance, int n_threads) {
    const size_t n = (size_t) j->w * j->h;
    rt3_dn_px* col[2] = { (rt3_dn_px*) aligned_alloc(16, n * sizeof(rt3_dn_px)), (rt3_dn_px*) aligned_alloc(16, n * sizeof(rt3_dn_px)) };
    rt3_dn_guide* guide = (rt3_dn_guide*) aligned_alloc(16, n * sizeof(rt3_dn_guide));
    if (!col[0] || !col[1] || !guide) { free(col[0]); free(col[1]); free(guide); return -1; }
    j->n_pow = (uint32_t) p->sigma_normal;
    j->gamma = !(flags & RT3_FLAG_NO_GAMMA);
    j->sigma_l = p->sigma_luminance; j->sigma_z = p->sigma_depth;
    j->guide = guide;
    j->in = NULL; j->out = col[1];
    for_each_row(j->h, n_threads, prepare, j);
    j->in = col[1]; j->out = col[0];
    for_each_row(j->h, n_threads, variance, j);
    for (uint32_t i = 0; i < p->iterations; i++) {
        j->in = col[i & 1u]; j->out = col[(i + 1u) & 1u];
        j->step = 1u << i;
        j->final_pass = i + 1u == p->iterations;
        for_each_row(j->h, n_threads, atrous_row, j);
    }
    free(col[0]); free(col[1]); free(guide);
    return 0;
}

const char* orc_denoise_check(const rt3_denoise_params* p) { return rt3_dn_check_params(p); }

const char* orc_denoise_temporal_check(const rt3_denoise_temporal_params* p) { return rt3_dn_check_temporal_params(p); }

/* The header's primitives over whole arrays, for their float64 checks (tests/test_denoise_reference.py): y = exp(-x),
 * y = b^n, and guide = (n^x, n^y, n^z, z) per pixel of normal [count][3] and depth [count]. */
void orc_dn_exp_neg(const float* x, float* y, size_t count) {
    for (size_t i = 0; i < count; i++) { y[i] = rt3_dn_exp_neg(x[i]); }
}

void orc_dn_pow(const float* b, const uint32_t* n_pow, float* y, size_t count) {
    for (size_t i = 0; i < count; i++) { y[i] = rt3_dn_pow(b[i], n_pow[i]); }
}

void orc_dn_make_guide(const float* normal, const float* depth, float* guide, size_t count) {
    for (size_t i = 0; i < count; i++) {
        const rt3_dn_guide g = rt3_dn_make_guide(normal[3 * i], normal[3 * i + 1], normal[3 * i + 2], depth[i]);
        guide[4 * i] = g.nx; guide[4 * i + 1] = g.ny; guide[4 * i + 2] = g.nz; guide[4 * i + 3] = g.z;
    }
}

/* The rays rt3_denoise_temporal reprojects: primary_ray of sample first_sample of every pixel, rays [h][w][6] (origin,
 * unit direction). */
void orc_dn_primary_rays(const rt3_camera* cam, const rt3_params* aov, float* rays) {
    for (uint32_t y = 0; y < aov->height; y++) {
        for (uint32_t x = 0; x < aov->width; x++) {
            v3 o, d = primary_ray(cam, aov, x, y, aov->first_sample, &o);
            float* r = rays + 6 * ((size_t) y * aov->width + x);
            r[0] = o.x; r[1] = o.y; r[2] = o.z; r[3] = d.x; r[4] = d.y; r[5] = d.z;
        }
    }
}

/* rt3_dn_reproject over `count` pixels: xy [count][2] pixel coordinates (integers), ray [count][6] origin and unit
 * direction, depth [count]; pos [count][4] = (x', y', |X - O_prev|, 1 when a position exists else 0). */
int orc_dn_reproject(const rt3_camera* cur, const rt3_camera* prev, uint32_t w, uint32_t h, const float* xy, const float* ray, const float* depth,
                     float* pos, size_t count) {
    for (size_t i = 0; i < count; i++) {
        const float* r = ray + 6 * i;
        float px = 0.0f, py = 0.0f, dist = 0.0f;
        const int ok = rt3_dn_reproject(*cur, *prev, w, h, (uint32_t) xy[2 * i], (uint32_t) xy[2 * i + 1], r[0], r[1], r[2], r[3], r[4], r[5], depth[i], &px,
                                        &py, &dist);
        pos[4 * i] = px; pos[4 * i + 1] = py; pos[4 * i + 2] = dist; pos[4 * i + 3] = (float) ok;
    }
    return 0;
}

int orc_denoise(uint32_t w, uint32_t h, const float* rgb, const float* albedo, const float* normal, const float* depth, const rt3_denoise_params* p,
                uint32_t flags, uint32_t* frame, float* rgb_out, int n_threads) {
    if (w < 1 || h < 1 || !rgb || !albedo || !normal || !depth || rt3_dn_check_params(p)) { return -1; }
    dn_job j = { .w = w, .h = h, .rgb = rgb, .albedo = albedo, .normal = normal, .depth = depth, .frame = frame, .rgb_out = rgb_out };
    return run_passes(&j, p, flags, prepare_row, variance_row, n_threads);
}

/* rt3_denoise_temporal on the host's arrays: rgb / albedo / normal / depth as orc_denoise takes them, the camera and the
 * parameters of the AOV call (its rays), and the previous history (read only when have_prev: its camera, per pixel colour
 * and length, moments and guide). Writes the next history, the frame, the linear rgb and the history length (either of
 * the last three may be NULL). */
int orc_denoise_temporal(uint32_t w, uint32_t h, const float* rgb, const float* albedo, const float* normal, const float* depth, const rt3_camera* cam,
                         const rt3_params* aov, const rt3_camera* prev_cam, int have_prev, const rt3_dn_hist* prev_col, const rt3_dn_moments* prev_mom,
                         const rt3_dn_guide* prev_guide, const rt3_denoise_temporal_params* tp, uint32_t flags, rt3_dn_hist* next_col,
                         rt3_dn_moments* next_mom, rt3_dn_guide* next_guide, uint32_t* frame, float* rgb_out, float* length, int n_threads) {
    if (w < 1 || h < 1 || !rgb || !albedo || !normal || !depth || !cam || !aov || !next_col || !next_mom || !next_guide || rt3_dn_check_temporal_params(tp)) {
        return -1;
    }
    if (have_prev && (!prev_cam || !prev_col || !prev_mom || !prev_guide)) { return -1; }
    dn_job j = { .w = w, .h = h, .rgb = rgb, .albedo = albedo, .normal = normal, .depth = depth, .frame = frame, .rgb_out = rgb_out,
                 .cam = cam, .prev_cam = prev_cam, .aov = aov, .have_prev = have_prev, .prev_col = prev_col, .prev_mom = prev_mom,
                 .prev_guide = prev_guide, .tp = tp, .next_col = next_col, .next_mom = next_mom, .next_guide = next_guide, .length = length };
    return run_passes(&j, &tp->filter, flags, temporal_row, temporal_variance_row, n_threads);
}
