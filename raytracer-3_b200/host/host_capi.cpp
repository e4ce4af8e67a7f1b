/* host_capi.cpp — C entry points over the C++ host backend, for the Python test harness.
 *
 * Drives the backend the way reference src/Main.cpp:266-288 drives any
 * Renderer: create entities through ECS::create_*, initialize_renderer(),
 * prerender(), Camera::update(), render(), read Camera::get_frame(). Every
 * call returns 0 or -1 (message in rt3host_last_error) where the C++ API would
 * throw CppDebugger::Fatal.
 */
#include <cstring>
#include <string>

#include <CppDebugger.hpp>

#include "entities/Triangle.hpp"
#include "entities/Sphere.hpp"
#include "entities/Object.hpp"
#include "renderer/CudaRenderer.hpp"
#include "sceneparser/SceneParser.hpp"

using namespace RayTracer;

namespace {
    struct HostScene {
        Tools::Array<ECS::RenderEntity*> entities;
        CudaRenderer* renderer = nullptr;
        Camera camera;
        ~HostScene() {
            for (size_t i = 0; i < entities.size(); i++) {
                /* entities are plain structs allocated by create_*; Object holds a std::string */
                if (entities[i]->type == ECS::et_object) { delete (ECS::Object*) entities[i]; }
                else if (entities[i]->type == ECS::et_sphere) { delete (ECS::Sphere*) entities[i]; }
                else { delete (ECS::Triangle*) entities[i]; }
            }
            delete renderer;
        }
    };
    thread_local std::string g_error;
    template <class F> int guarded(F&& body) {
        try { body(); return 0; }
        catch (std::exception& e) { g_error = e.what(); return -1; }
    }
    glm::vec3 v3(const float* p) { return glm::vec3(p[0], p[1], p[2]); }
}

extern "C" {

const char* rt3host_last_error() { return g_error.c_str(); }
void* rt3host_scene_create() { return new HostScene(); }
void rt3host_scene_destroy(void* s) { delete (HostScene*) s; }

int rt3host_add_triangle(void* s, const float* p1, const float* p2, const float* p3, const float* color) {
    return guarded([&] { ((HostScene*) s)->entities.push_back(ECS::create_triangle(v3(p1), v3(p2), v3(p3), v3(color))); });
}
int rt3host_add_sphere(void* s, const float* center, float radius, uint32_t n_meridians, uint32_t n_parallels, const float* color) {
    return guarded([&] { ((HostScene*) s)->entities.push_back(ECS::create_sphere(v3(center), radius, n_meridians, n_parallels, v3(color))); });
}
int rt3host_add_object(void* s, const char* path, const float* center, float scale, const float* color) {
    return guarded([&] { ((HostScene*) s)->entities.push_back(ECS::create_object(path, v3(center), scale, v3(color))); });
}

/* SceneLang front end: appends the entities of a .scene text to the scene; returns how many were added through *n_added
 * and the warnings (newline separated) through rt3host_last_error when there are any. */
int rt3host_add_scene_text(void* s, const char* text, const char* base_dir, uint32_t* n_added) {
    HostScene* hs = (HostScene*) s;
    return guarded([&] {
        ParsedScene parsed;
        SceneParser::parse_string(text, base_dir ? base_dir : "", parsed);
        for (size_t i = 0; i < parsed.entities.size(); i++) { hs->entities.push_back(parsed.entities[i]); }
        if (n_added) { *n_added = (uint32_t) parsed.entities.size(); }
        g_error.clear();
        for (const std::string& w : parsed.warnings) { g_error += w + "\n"; }
    });
}

/* CPU-only flatten of one entity list (no device needed): the arrays prerender() would upload. */
int rt3host_flatten(void* s, uint32_t* n_faces, uint32_t* n_vertices, void* faces_out, void* vertices_out, uint32_t* face_entity_out) {
    HostScene* hs = (HostScene*) s;
    return guarded([&] {
        Tools::Array<GFace> faces;
        Tools::Array<glm::vec4> vertices;
        uint32_t nf = 0, nv = 0;
        for (size_t i = 0; i < hs->entities.size(); i++) {
            ECS::RenderEntity* e = hs->entities[i];
            faces.clear(); vertices.clear();
            faces.resize(e->pre_render_faces); vertices.resize(e->pre_render_vertices);
            if (e->type == ECS::et_triangle) { ECS::cpu_pre_render_triangle(faces, vertices, (ECS::Triangle*) e); }
            else if (e->type == ECS::et_sphere) { ECS::cpu_pre_render_sphere(faces, vertices, (ECS::Sphere*) e); }
            else { ECS::cpu_pre_render_object(faces, vertices, (ECS::Object*) e); }
            for (size_t f = 0; f < faces.size(); f++) {
                if (faces_out) {
                    GFace g = faces[f];
                    g.v1 += nv; g.v2 += nv; g.v3 += nv;
                    std::memcpy((char*) faces_out + 48 * (size_t) (nf + f), &g, 48);
                }
                if (face_entity_out) { face_entity_out[nf + f] = (uint32_t) i; }
            }
            if (vertices_out) { for (size_t v = 0; v < vertices.size(); v++) { std::memcpy((char*) vertices_out + 16 * (size_t) (nv + v), &vertices[v], 16); } }
            nf += (uint32_t) faces.size(); nv += (uint32_t) vertices.size();
        }
        *n_faces = nf; *n_vertices = nv;
    });
}

/* The flattened scene the renderer holds after prerender() (CudaRenderer::flat_faces / flat_vertices): with
 * device_tessellation these are read back from the device arrays the kernels filled. Sizes first (NULL outputs), then the data. */
int rt3host_renderer_flat(void* s, uint32_t* n_faces, uint32_t* n_vertices, void* faces_out, void* vertices_out) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    *n_faces = (uint32_t) hs->renderer->flat_faces.size(); *n_vertices = (uint32_t) hs->renderer->flat_vertices.size();
    if (faces_out) { std::memcpy(faces_out, hs->renderer->flat_faces.data(), sizeof(rt3_face) * hs->renderer->flat_faces.size()); }
    if (vertices_out) { std::memcpy(vertices_out, hs->renderer->flat_vertices.data(), sizeof(rt3_vertex) * hs->renderer->flat_vertices.size()); }
    return 0;
}

/* initialize_renderer() + settings; mode 0 = reference, 1 = pathtrace. */
int rt3host_renderer_create(void* s, int device, uint32_t mode, uint32_t spp, uint32_t max_depth, uint32_t seed, uint32_t flags, int analytic_spheres) {
    HostScene* hs = (HostScene*) s;
    return guarded([&] {
        delete hs->renderer;
        hs->renderer = nullptr;
        hs->renderer = new CudaRenderer(device);
        CudaRenderSettings st;
        st.mode = mode; st.spp = spp; st.max_depth = max_depth; st.seed = seed; st.flags = flags;
        st.analytic_spheres = (analytic_spheres & 1) != 0; st.device_tessellation = (analytic_spheres & 2) != 0; /* bit 0 / bit 1 */
        hs->renderer->set_settings(st);
    });
}
/* The same over several devices (one context each, CudaRenderer(const std::vector<int>&)); a device may be listed twice. */
int rt3host_renderer_create_multi(void* s, const int* devices, uint32_t n_devices, uint32_t mode, uint32_t spp, uint32_t max_depth, uint32_t seed,
                                  uint32_t flags, int analytic_spheres, uint32_t tile_rows) {
    HostScene* hs = (HostScene*) s;
    return guarded([&] {
        delete hs->renderer;
        hs->renderer = nullptr;
        hs->renderer = new CudaRenderer(std::vector<int>(devices, devices + n_devices));
        CudaRenderSettings st;
        st.mode = mode; st.spp = spp; st.max_depth = max_depth; st.seed = seed; st.flags = flags;
        st.analytic_spheres = (analytic_spheres & 1) != 0; st.device_tessellation = (analytic_spheres & 2) != 0;
        if (tile_rows) { st.tile_rows = tile_rows; }
        hs->renderer->set_settings(st);
    });
}
int rt3host_set_material(void* s, uint32_t entity_index, uint32_t kind, const float* albedo, float fuzz, float ior) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    Material m;
    m.kind = (Material::Kind) kind; m.albedo = v3(albedo); m.fuzz = fuzz; m.ior = ior;
    hs->renderer->set_material(entity_index, m);
    return 0;
}
int rt3host_prerender(void* s) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] { hs->renderer->prerender(hs->entities); });
}
/* Camera::update(W, H, focal, vw, vh) (reference Main.cpp:272) or look_at when from_at_up_vfov_aperture_focus != NULL (12 floats). */
int rt3host_render(void* s, uint32_t width, uint32_t height, float focal, float vw, float vh, const float* look, uint32_t* frame_out, double* device_ms,
                   uint64_t* rays) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] {
        if (look) { hs->camera.look_at(width, height, v3(look), v3(look + 3), v3(look + 6), look[9], look[10], look[11]); }
        else { hs->camera.update(width, height, focal, vw, vh); }
        hs->renderer->render(hs->camera);
        std::memcpy(frame_out, hs->camera.get_frame().d(), sizeof(uint32_t) * (size_t) width * height);
        if (device_ms) { *device_ms = hs->renderer->stats().device_ms; }
        if (rays) { *rays = hs->renderer->stats().rays; }
    });
}
/* CudaRenderer::render_progressive with the reference camera; frames_out receives every pass's frame (passes * W * H words). */
int rt3host_render_progressive(void* s, uint32_t width, uint32_t height, float focal, float vw, float vh, uint32_t passes, uint32_t* frames_out) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] {
        hs->camera.update(width, height, focal, vw, vh);
        struct Sink { uint32_t* out; size_t n; } sink = { frames_out, (size_t) width * height };
        hs->renderer->render_progressive(hs->camera, passes, [](uint32_t pass, const Frame& f, void* user) {
            Sink* k = (Sink*) user;
            std::memcpy(k->out + (size_t) pass * k->n, f.d(), sizeof(uint32_t) * k->n);
        }, &sink);
    });
}
/* CudaRenderer::read_radiance of the last render (rgb_out: width * height * 3 floats) and, if path != NULL, write_radiance_pfm. */
int rt3host_radiance(void* s, uint32_t width, uint32_t height, float* rgb_out, const char* path) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] {
        if (rgb_out) {
            std::vector<float> rgb;
            hs->renderer->read_radiance(width, height, rgb);
            std::memcpy(rgb_out, rgb.data(), rgb.size() * sizeof(float));
        }
        if (path) { hs->renderer->write_radiance_pfm(width, height, path); }
    });
}
/* CudaRenderer::render_path_aovs with the reference camera and settings.aov_spp = aov_spp (out: host arrays of width * height
 * pixels, any may be NULL) and, if dir != NULL, write_path_aovs_pfm into dir. */
int rt3host_path_aovs(void* s, uint32_t width, uint32_t height, float focal, float vw, float vh, uint32_t aov_spp, const rt3_path_aovs* out, const char* dir) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] {
        hs->camera.update(width, height, focal, vw, vh);
        CudaRenderSettings st = hs->renderer->get_settings();
        st.aov_spp = aov_spp;
        hs->renderer->set_settings(st);
        CudaPathAovs aovs;
        hs->renderer->render_path_aovs(hs->camera, aovs);
        if (out) {
            const size_t n = (size_t) width * height;
            if (out->hit_prim) { std::memcpy(out->hit_prim, aovs.hit_prim.data(), n * sizeof(uint32_t)); }
            if (out->hit_entity) { std::memcpy(out->hit_entity, aovs.hit_entity.data(), n * sizeof(uint32_t)); }
            if (out->hit_t) { std::memcpy(out->hit_t, aovs.hit_t.data(), n * sizeof(float)); }
            if (out->albedo) { std::memcpy(out->albedo, aovs.albedo.data(), 3 * n * sizeof(float)); }
            if (out->normal) { std::memcpy(out->normal, aovs.normal.data(), 3 * n * sizeof(float)); }
        }
        if (dir) { hs->renderer->write_path_aovs_pfm(aovs, dir); }
    });
}
/* CudaRenderer::denoise with the reference camera (frame_out: width * height words, rgb_out: width * height * 3 floats; either may be NULL). */
int rt3host_denoise(void* s, uint32_t width, uint32_t height, float focal, float vw, float vh, const rt3_denoise_params* p, uint32_t* frame_out, float* rgb_out) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] {
        hs->camera.update(width, height, focal, vw, vh);
        CudaDenoiseSettings st;
        st.iterations = p->iterations; st.sigma_luminance = p->sigma_luminance; st.sigma_normal = p->sigma_normal; st.sigma_depth = p->sigma_depth;
        std::vector<float> rgb;
        hs->renderer->denoise(hs->camera, st, rgb_out ? &rgb : nullptr);
        if (frame_out) { std::memcpy(frame_out, hs->camera.get_frame().d(), (size_t) width * height * sizeof(uint32_t)); }
        if (rgb_out) { std::memcpy(rgb_out, rgb.data(), rgb.size() * sizeof(float)); }
    });
}
/* CudaRenderer::denoise_temporal with the reference camera (outputs as rt3host_denoise's). */
int rt3host_denoise_temporal(void* s, uint32_t width, uint32_t height, float focal, float vw, float vh, const rt3_denoise_temporal_params* p, uint32_t* frame_out,
                             float* rgb_out) {
    HostScene* hs = (HostScene*) s;
    if (!hs->renderer) { g_error = "create the renderer first"; return -1; }
    return guarded([&] {
        hs->camera.update(width, height, focal, vw, vh);
        CudaDenoiseTemporalSettings st;
        st.filter.iterations = p->filter.iterations; st.filter.sigma_luminance = p->filter.sigma_luminance;
        st.filter.sigma_normal = p->filter.sigma_normal; st.filter.sigma_depth = p->filter.sigma_depth;
        st.alpha_color = p->alpha_color; st.alpha_moments = p->alpha_moments; st.depth_tolerance = p->depth_tolerance; st.normal_cos = p->normal_cos;
        std::vector<float> rgb;
        hs->renderer->denoise_temporal(hs->camera, st, p->reset != 0, rgb_out ? &rgb : nullptr);
        if (frame_out) { std::memcpy(frame_out, hs->camera.get_frame().d(), (size_t) width * height * sizeof(uint32_t)); }
        if (rgb_out) { std::memcpy(rgb_out, rgb.data(), rgb.size() * sizeof(float)); }
    });
}
int rt3host_camera_vectors(uint32_t width, uint32_t height, const float* look, float* out19) {
    return guarded([&] {
        Camera cam;
        cam.look_at(width, height, v3(look), v3(look + 3), v3(look + 6), look[9], look[10], look[11]);
        const glm::vec3* v[6] = { &cam.origin, &cam.horizontal, &cam.vertical, &cam.lower_left_corner, &cam.lens_u, &cam.lens_v };
        for (int i = 0; i < 4; i++) { out19[3 * i] = v[i]->x; out19[3 * i + 1] = v[i]->y; out19[3 * i + 2] = v[i]->z; }
        out19[12] = cam.lens_radius;
        for (int i = 4; i < 6; i++) { out19[13 + 3 * (i - 4)] = v[i]->x; out19[14 + 3 * (i - 4)] = v[i]->y; out19[15 + 3 * (i - 4)] = v[i]->z; }
    });
}

/* Frame::to_png / Frame::to_ppm on a caller-supplied frame (format: 0 = PPM, 1 = PNG). */
int rt3host_write_image(const uint32_t* frame, uint32_t width, uint32_t height, const char* path, int format) {
    return guarded([&] {
        Frame f(width, height);
        std::memcpy(f.d(), frame, sizeof(uint32_t) * (size_t) width * height);
        if (format == 1) { f.to_png(path); } else { f.to_ppm(path); }
    });
}

}  // extern "C"
