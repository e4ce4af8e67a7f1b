/* denoise_oracle.c — CPU restatement of rt3_denoise (TEST INFRASTRUCTURE, plain C11, built by tests/denoise_lib.py with the
 * oracle's flags: -O2 -ffp-contract=off -fno-fast-math).
 *
 * The filter's arithmetic is include/rt3_denoise.h, the same functions the kernels call; this file restates only what the
 * kernels do around them: the order of the passes, the ping-pong buffers and the resolve (resolve_kernel's gamma, unorm8
 * and packing; the oracle's unorm8 is the kernels'). Its inputs are the arrays rt3_read_radiance and rt3_render_path_aovs
 * return, so it can be fed the GPU's own inputs, or synthetic ones. The oracle is compiled into this unit for its row pool
 * (for_each_row) and unorm8. Any width and height >= 1 are accepted (the library renders nothing under 2x2). */
#include "../oracle/rt3_oracle.c"
#include "rt3_denoise.h"

int orc_denoise(uint32_t w, uint32_t h, const float* rgb, const float* albedo, const float* normal, const float* depth, const rt3_denoise_params* p,
                uint32_t flags, uint32_t* frame, float* rgb_out, int n_threads);
const char* orc_denoise_check(const rt3_denoise_params* p);
void orc_dn_exp_neg(const float* x, float* y, size_t count);
void orc_dn_pow(const float* b, const uint32_t* n_pow, float* y, size_t count);
void orc_dn_make_guide(const float* normal, const float* depth, float* guide, size_t count);

typedef struct {
    uint32_t w, h, step, n_pow, final_pass, gamma;
    float sigma_l, sigma_z;
    const float *rgb, *albedo, *normal, *depth;
    rt3_dn_px *in, *out;
    rt3_dn_guide* guide;
    uint32_t* frame;
    float* rgb_out;
} dn_job;

static void prepare_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        rt3_dn_prepare_px(j->rgb + 3 * i, j->albedo + 3 * i, j->normal + 3 * i, j->depth[i], &j->out[i], &j->guide[i]);
    }
}

static void variance_row(void* ctx, uint32_t y) {
    const dn_job* j = (const dn_job*) ctx;
    for (uint32_t x = 0; x < j->w; x++) {
        const size_t i = (size_t) y * j->w + x;
        j->out[i] = j->in[i];
        j->out[i].v = rt3_dn_variance_px(j->in, j->guide, j->w, j->h, x, y, j->sigma_z, j->n_pow);
    }
}

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

const char* orc_denoise_check(const rt3_denoise_params* p) { return rt3_dn_check_params(p); }

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

int orc_denoise(uint32_t w, uint32_t h, const float* rgb, const float* albedo, const float* normal, const float* depth, const rt3_denoise_params* p,
                uint32_t flags, uint32_t* frame, float* rgb_out, int n_threads) {
    if (w < 1 || h < 1 || !rgb || !albedo || !normal || !depth || rt3_dn_check_params(p)) { return -1; }
    const size_t n = (size_t) w * h;
    rt3_dn_px* col[2] = { (rt3_dn_px*) aligned_alloc(16, n * sizeof(rt3_dn_px)), (rt3_dn_px*) aligned_alloc(16, n * sizeof(rt3_dn_px)) };
    rt3_dn_guide* guide = (rt3_dn_guide*) aligned_alloc(16, n * sizeof(rt3_dn_guide));
    if (!col[0] || !col[1] || !guide) { free(col[0]); free(col[1]); free(guide); return -1; }
    dn_job j = { w, h, 0, (uint32_t) p->sigma_normal, 0, !(flags & RT3_FLAG_NO_GAMMA), p->sigma_luminance, p->sigma_depth,
                 rgb, albedo, normal, depth, NULL, col[1], guide, frame, rgb_out };
    for_each_row(h, n_threads, prepare_row, &j);
    j.in = col[1]; j.out = col[0];
    for_each_row(h, n_threads, variance_row, &j);
    for (uint32_t i = 0; i < p->iterations; i++) {
        j.in = col[i & 1u]; j.out = col[(i + 1u) & 1u];
        j.step = 1u << i;
        j.final_pass = i + 1u == p->iterations;
        for_each_row(h, n_threads, atrous_row, &j);
    }
    free(col[0]); free(col[1]); free(guide);
    return 0;
}
