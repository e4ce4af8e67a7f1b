/* path_aov_oracle.c — CPU restatement of rt3_render_path_aovs (TEST INFRASTRUCTURE, plain C11, built by
 * tests/path_aov_lib.py with the oracle's flags: -O2 -ffp-contract=off -fno-fast-math).
 *
 * The AOVs are those of the path tracer's primary rays, so they must come from the oracle's own closest-hit tests and
 * material lookup. The oracle (oracle/rt3_oracle.c) is compiled into this unit as it is, which gives the code below its
 * closest_face, closest_sphere_path, material_of and prim_entity without a second copy of them and without a change to
 * the pinned file. Only the ray set-up of trace_path's first segment is restated (primary_ray).
 *
 * Semantics (include/rt3cuda.h, DESIGN.md 3.7): for the samples [first_sample, first_sample + spp) of every owned pixel,
 * the albedo the path tracer multiplies by at the first hit (dielectric 1, miss: the sky with throughput 1) and the
 * front-facing normal (miss 0), summed in 2^24 fixed point and resolved as the radiance is; hit_prim / hit_entity / hit_t
 * of sample first_sample. */
#include "../oracle/rt3_oracle.c"

int orc_render_path_aovs(const rt3_scene* scene, const rt3_camera* cam, const rt3_params* p, const rt3_path_aovs* out, int n_threads);

/* trace_path's primary ray of (x, y, sample): origin in *o, unit direction returned. */
static v3 primary_ray(const rt3_camera* cam, const rt3_params* p, uint32_t x, uint32_t y, uint32_t sample, v3* o_out) {
    uint32_t pixel_index = y * p->width + x;
    uint32_t key = rt3_path_key(pixel_index, sample, p->seed);
    float jx = 0.0f, jy = 0.0f;
    if (!(p->flags & RT3_FLAG_NO_JITTER)) { jx = rt3_draw(key, RT3_DIM_JITTER_X); jy = rt3_draw(key, RT3_DIM_JITTER_Y); }
    float u = ((float) x + jx) / ((float) p->width - 1.0f);
    float v = ((float) (p->height - 1 - y) + jy) / ((float) p->height - 1.0f);
    v3 o = vld(cam->origin);
    v3 dir = vsub(vadd(vadd(vld(cam->lower_left_corner), vscale(u, vld(cam->horizontal))), vscale(v, vld(cam->vertical))), o);
    if (cam->lens_radius > 0.0f) {
        float r = sqrtf(rt3_draw(key, RT3_DIM_LENS_R));
        float sn, cs;
        rt3_sincos_2pi(rt3_draw(key, RT3_DIM_LENS_PHI), &sn, &cs);
        float lx = cam->lens_radius * (r * cs), ly = cam->lens_radius * (r * sn);
        v3 off = vadd(vscale(lx, vld(cam->lens_u)), vscale(ly, vld(cam->lens_v)));
        o = vadd(o, off);
        dir = vsub(dir, off);
    }
    *o_out = o;
    return normalize3(dir);
}

/* Signed 2^24 fixed point: round to nearest even, clamped to +-2^20, NaN -> 0. */
static inline int64_t to_fixed_signed(float c) {
    float s = c * RT3_ACC_SCALE;
    if (s != s) { return 0; }
    if (s < -17592186044416.0f) { s = -17592186044416.0f; }
    if (s > 17592186044416.0f) { s = 17592186044416.0f; }
    return (int64_t) llrintf(s);
}

#define AOV_XBLOCK 64u /* pixels of a row per work unit: a one-row partition still uses every thread */

typedef struct { const rt3_scene* scene; const rt3_camera* cam; const rt3_params* p; const rt3_path_aovs* out; uint32_t xblocks; } aov_job;

static void path_aov_unit(void* ctx, uint32_t unit) {
    const aov_job* j = (const aov_job*) ctx;
    const rt3_scene* s = j->scene; const rt3_params* p = j->p; const rt3_path_aovs* out = j->out;
    const uint32_t y = unit / j->xblocks, x0 = (unit % j->xblocks) * AOV_XBLOCK;
    const uint32_t tile_rows = p->tile_rows ? p->tile_rows : 1, parts = p->part_count ? p->part_count : 1;
    if ((y / tile_rows) % parts != p->part_index % parts) { return; }
    const uint32_t x1 = x0 + AOV_XBLOCK < p->width ? x0 + AOV_XBLOCK : p->width;
    for (uint32_t x = x0; x < x1; x++) {
        uint64_t alb[3] = { 0, 0, 0 }, nrm[3] = { 0, 0, 0 }; /* the normal sums in two's complement, as on the device */
        const size_t idx = (size_t) y * p->width + x;
        for (uint32_t sidx = 0; sidx < p->spp; sidx++) {
            v3 o, d = primary_ray(j->cam, p, x, y, p->first_sample + sidx, &o);
            hit_rec best = { NO_HIT, INFINITY };
            best = closest_face(s, o, d, RT3_TMIN, best);
            best = closest_sphere_path(s, o, d, best);
            v3 albedo, n = V(0.0f, 0.0f, 0.0f);
            if (best.prim == NO_HIT) {
                if (p->flags & RT3_FLAG_UNIFORM_SKY) { albedo = V(1.0f, 1.0f, 1.0f); }
                else {
                    float t = 0.5f * (d.y + 1.0f);
                    float a = 1.0f - t;
                    albedo = V(a * 1.0f + t * 0.5f, a * 1.0f + t * 0.7f, a * 1.0f + t * 1.0f);
                }
            } else {
                v3 hp = vadd(o, vscale(best.t, d));
                v3 outward;
                if (best.prim < s->n_faces) {
                    outward = vld(s->faces[best.prim].normal);
                } else {
                    const rt3_sphere* sp = &s->spheres[best.prim - s->n_faces];
                    v3 pc = vsub(hp, V(sp->cx, sp->cy, sp->cz));
                    outward = V(pc.x / sp->r, pc.y / sp->r, pc.z / sp->r);
                }
                n = dot3(d, outward) < 0.0f ? outward : vneg(outward);
                rt3_material m;
                material_of(s, best.prim, &m);
                albedo = m.kind == RT3_MAT_DIELECTRIC ? V(1.0f, 1.0f, 1.0f) : vld(m.albedo);
            }
            alb[0] += to_fixed(albedo.x); alb[1] += to_fixed(albedo.y); alb[2] += to_fixed(albedo.z);
            nrm[0] += (uint64_t) to_fixed_signed(n.x); nrm[1] += (uint64_t) to_fixed_signed(n.y); nrm[2] += (uint64_t) to_fixed_signed(n.z);
            if (sidx == 0) {
                if (out->hit_prim) { out->hit_prim[idx] = best.prim; }
                if (out->hit_entity) { out->hit_entity[idx] = prim_entity(s, best.prim); }
                if (out->hit_t) { out->hit_t[idx] = best.t; }
            }
        }
        const double scale = (double) p->spp * (double) RT3_ACC_SCALE;
        for (int c = 0; c < 3; c++) {
            if (out->albedo) { out->albedo[3 * idx + c] = (float) ((double) alb[c] / scale); }
            if (out->normal) { out->normal[3 * idx + c] = (float) ((double) (int64_t) nrm[c] / scale); }
        }
    }
}

int orc_render_path_aovs(const rt3_scene* scene, const rt3_camera* cam, const rt3_params* p, const rt3_path_aovs* out, int n_threads) {
    if (!scene || !cam || !p || !out || p->width < 2 || p->height < 2 || p->spp < 1) { return -1; }
    aov_job job = { scene, cam, p, out, (p->width + AOV_XBLOCK - 1) / AOV_XBLOCK };
    for_each_row(p->height * job.xblocks, n_threads, path_aov_unit, &job);
    return 0;
}
