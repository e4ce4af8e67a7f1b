/* renderer/CudaRenderer.cpp — see CudaRenderer.hpp. */
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include <CppDebugger.hpp>

#include "entities/Triangle.hpp"
#include "entities/Sphere.hpp"
#include "entities/Object.hpp"

#include "CudaRenderer.hpp"

using namespace RayTracer;
using namespace RayTracer::ECS;
using namespace CppDebugger::SeverityValues;

static_assert(sizeof(GFace) == sizeof(rt3_face), "GFace and rt3_face must share a layout");
static_assert(sizeof(glm::vec4) == sizeof(rt3_vertex), "vec4 and rt3_vertex must share a layout");

namespace {
    void check(int status, const char* what) {
        if (status != RT3_OK) { DLOG(fatal, std::string(what) + ": " + rt3_last_error()); }
    }

    uint32_t env_u32(const char* name, uint32_t fallback) {
        const char* v = std::getenv(name);
        return (v && *v) ? (uint32_t) std::strtoul(v, nullptr, 0) : fallback;
    }
}

CudaRenderSettings CudaRenderSettings::from_environment(int* device) {
    CudaRenderSettings s;
    const char* mode = std::getenv("RT3_MODE");
    if (mode && std::string(mode) == "pathtrace") { s.mode = RT3_MODE_PATHTRACE; }
    s.spp = env_u32("RT3_SPP", s.spp);
    s.max_depth = env_u32("RT3_DEPTH", s.max_depth);
    s.seed = env_u32("RT3_SEED", s.seed);
    s.analytic_spheres = env_u32("RT3_ANALYTIC_SPHERES", 0) != 0;
    s.device_tessellation = env_u32("RT3_DEVICE_TESSELLATION", 0) != 0;
    s.bvh_above = env_u32("RT3_BVH_ABOVE", s.bvh_above);
    if (env_u32("RT3_BVH", 0) != 0) { s.flags |= RT3_FLAG_BVH; }
    if (device) { *device = (int) env_u32("RT3_DEVICE", 0); }
    return s;
}

std::vector<int> CudaRenderSettings::devices_from_environment() {
    std::vector<int> out;
    const char* v = std::getenv("RT3_DEVICES");
    if (v && std::string(v) == "all") {
        /* as many as rt3_create accepts */
        for (int d = 0; d < 64; d++) {
            rt3_ctx* probe = nullptr;
            if (rt3_create(&probe, d) != RT3_OK) { break; }
            rt3_destroy(probe);
            out.push_back(d);
        }
    } else if (v && *v) {
        const char* p = v;
        while (*p) {
            char* end = nullptr;
            long d = std::strtol(p, &end, 10);
            if (end == p) { break; }
            out.push_back((int) d);
            p = (*end == ',') ? end + 1 : end;
            if (*end != ',' && *end != '\0') { break; }
        }
    }
    if (out.empty()) { out.push_back((int) env_u32("RT3_DEVICE", 0)); }
    return out;
}

CudaRenderer::CudaRenderer(int device) : Renderer(), ctx(nullptr), shared_frame(nullptr), shared_pixels(0) {
    std::memset(&this->last_stats, 0, sizeof this->last_stats);
    check(rt3_create(&this->ctx, device), "Could not create the CUDA render context");
}

CudaRenderer::CudaRenderer(const std::vector<int>& devices) : Renderer(), ctx(nullptr), shared_frame(nullptr), shared_pixels(0) {
    std::memset(&this->last_stats, 0, sizeof this->last_stats);
    if (devices.empty()) { DLOG(fatal, "CudaRenderer needs at least one device."); }
    check(rt3_create(&this->ctx, devices[0]), "Could not create the CUDA render context");
    for (size_t i = 1; i < devices.size(); i++) {
        rt3_ctx* helper = nullptr;
        int rc = rt3_create(&helper, devices[i]);
        if (rc == RT3_OK) {
            this->helpers.push_back(helper);
            rc = rt3_frame_attach(helper, this->ctx);
        }
        if (rc != RT3_OK) {
            const std::string why = rt3_last_error();
            this->release();
            DLOG(fatal, "Could not set up device " + std::to_string(devices[i]) + ": " + why);
        }
    }
}

void CudaRenderer::release() noexcept {
    /* helpers first: rt3_destroy waits for their streams, and their kernels store into the shared frame over NVLink --
     * it may only be freed once nothing can write to it any more (a render that failed half-way leaves work enqueued) */
    for (size_t i = 0; i < this->helpers.size(); i++) { rt3_destroy(this->helpers[i]); }
    this->helpers.clear();
    if (this->shared_frame) { rt3_frame_free(this->ctx, this->shared_frame); this->shared_frame = nullptr; this->shared_pixels = 0; }
    rt3_destroy(this->ctx);
    this->ctx = nullptr;
}

CudaRenderer::~CudaRenderer() { this->release(); }

void CudaRenderer::prerender(const Tools::Array<ECS::RenderEntity*>& entities) {
    this->flat_faces.clear(); this->flat_vertices.clear(); this->flat_face_entity.clear(); this->flat_spheres.clear();
    std::vector<uint32_t> face_material, sphere_material, sphere_entity;
    std::vector<float> sphere_color;
    std::vector<rt3_material> table;
    bool any_material = !this->materials.empty();

    /* device scene (settings.device_tessellation): spheres are tessellated on the device straight into the flattened arrays
     * there; the host arrays keep zeroed placeholders for them (so that offsets are the reference's) and are filled from the
     * device afterwards for inspection. `host_ranges` are the stretches the host did produce (triangles, object files). */
    struct DeferredSphere { rt3_uv_sphere d; uint32_t first_vertex, first_face; };
    struct Range { size_t first_face, n_faces, first_vertex, n_vertices; };
    std::vector<DeferredSphere> deferred;
    std::vector<Range> host_ranges;
    const bool device_scene = this->settings.device_tessellation;

    Tools::Array<GFace> faces;
    Tools::Array<glm::vec4> vertices;
    for (size_t i = 0; i < entities.size(); i++) {
        RenderEntity* e = entities[i];
        if (!(e->pre_render_mode & EntityPreRenderModeFlags::eprmf_cpu)) {
            DLOG(fatal, "Entity " + std::to_string(i) + " of type " + entity_type_names[e->type] + " cannot be pre-rendered on the CPU.");
        }
        /* material row of this entity: explicit, or Lambertian(colour) when any material is in use */
        uint32_t material_index = 0;
        glm::vec3 entity_color(1.0f, 1.0f, 1.0f);
        switch (e->pre_render_operation) {
            case EntityPreRenderOperation::epro_generate_triangle: entity_color = ((Triangle*) e)->color; break;
            case EntityPreRenderOperation::epro_generate_sphere: entity_color = ((Sphere*) e)->color; break;
            case EntityPreRenderOperation::epro_load_object_file: entity_color = ((Object*) e)->color; break;
            default: break;
        }
        if (any_material) {
            Material m;
            m.albedo = entity_color;
            std::map<size_t, Material>::const_iterator it = this->materials.find(i);
            if (it != this->materials.end()) { m = it->second; }
            rt3_material row;
            std::memset(&row, 0, sizeof row);
            row.kind = (uint32_t) m.kind;
            row.albedo[0] = m.albedo.x; row.albedo[1] = m.albedo.y; row.albedo[2] = m.albedo.z;
            row.fuzz = m.fuzz; row.ior = m.ior;
            material_index = (uint32_t) table.size();
            table.push_back(row);
        }

        if (e->pre_render_operation == EntityPreRenderOperation::epro_generate_sphere && this->settings.analytic_spheres) {
            const Sphere* s = (const Sphere*) e;
            rt3_sphere sp = { s->center.x, s->center.y, s->center.z, s->radius };
            this->flat_spheres.push_back(sp);
            sphere_color.push_back(s->color.x); sphere_color.push_back(s->color.y); sphere_color.push_back(s->color.z);
            sphere_entity.push_back((uint32_t) i);
            sphere_material.push_back(material_index);
            continue;
        }

        /* tessellate / load into per-entity buffers of the announced size (SequentialRenderer.cpp:216-243) */
        faces.clear(); vertices.clear();
        faces.resize(e->pre_render_faces);
        vertices.resize(e->pre_render_vertices);
        switch (e->pre_render_operation) {
            case EntityPreRenderOperation::epro_generate_triangle: cpu_pre_render_triangle(faces, vertices, (Triangle*) e); break;
            case EntityPreRenderOperation::epro_generate_sphere:
                if (device_scene) {
                    /* the reference's GPU pre-render (VulkanRenderer.cpp:310-336) as a CUDA kernel, CPU-path arithmetic; run after
                     * this loop, when the device arrays exist */
                    const Sphere* sp = (const Sphere*) e;
                    DeferredSphere job = { { { sp->center.x, sp->center.y, sp->center.z }, sp->radius, sp->n_meridians, sp->n_parallels,
                                             { sp->color.x, sp->color.y, sp->color.z }, (uint32_t) i },
                                           (uint32_t) this->flat_vertices.size(), (uint32_t) this->flat_faces.size() };
                    deferred.push_back(job);
                    std::memset((void*) &faces[0], 0, faces.size() * sizeof(GFace));
                    std::memset((void*) &vertices[0], 0, vertices.size() * sizeof(glm::vec4));
                } else {
                    cpu_pre_render_sphere(faces, vertices, (Sphere*) e);
                }
                break;
            case EntityPreRenderOperation::epro_load_object_file: cpu_pre_render_object(faces, vertices, (Object*) e); break;
            default:
                DLOG(fatal, "Entity " + std::to_string(i) + " wants to be pre-rendered using unsupported operation '" +
                                entity_pre_render_operation_names[e->pre_render_operation] + "'.");
        }
        if (device_scene && e->pre_render_operation != EntityPreRenderOperation::epro_generate_sphere) {
            Range r = { this->flat_faces.size(), faces.size(), this->flat_vertices.size(), vertices.size() };
            host_ranges.push_back(r);
        }
        /* append with re-based indices (SequentialRenderer.cpp:174-195) */
        const uint32_t offset = (uint32_t) this->flat_vertices.size();
        for (size_t f = 0; f < faces.size(); f++) {
            rt3_face out;
            std::memcpy(&out, &faces[f], sizeof out);
            out.v1 += offset; out.v2 += offset; out.v3 += offset;
            this->flat_faces.push_back(out);
            this->flat_face_entity.push_back((uint32_t) i);
            face_material.push_back(material_index);
        }
        for (size_t v = 0; v < vertices.size(); v++) {
            rt3_vertex out;
            std::memcpy(&out, &vertices[v], sizeof out);
            this->flat_vertices.push_back(out);
        }
    }

    rt3_scene scene;
    std::memset(&scene, 0, sizeof scene);
    scene.n_faces = (uint32_t) this->flat_faces.size();
    scene.n_vertices = (uint32_t) this->flat_vertices.size();
    scene.faces = this->flat_faces.data();
    scene.vertices = this->flat_vertices.data();
    scene.face_entity = this->flat_face_entity.data();
    scene.face_material = any_material ? face_material.data() : nullptr;
    scene.n_spheres = (uint32_t) this->flat_spheres.size();
    scene.spheres = this->flat_spheres.data();
    scene.sphere_color = sphere_color.data();
    scene.sphere_entity = sphere_entity.data();
    scene.sphere_material = any_material ? sphere_material.data() : nullptr;
    scene.n_materials = (uint32_t) table.size();
    scene.materials = table.data();
    if (!device_scene) {
        check(rt3_scene_upload(this->ctx, &scene), "Could not upload the scene");
        for (size_t i = 0; i < this->helpers.size(); i++) { check(rt3_scene_upload(this->helpers[i], &scene), "Could not upload the scene to a further device"); }
        return;
    }

    /* Device scene: the flattened arrays are assembled in each device's memory -- the host's stretches by plain copies, the
     * spheres by the tessellation kernels -- and everything derived from them is built there (rt3_scene_upload_device). */
    struct DeviceArrays {
        rt3_ctx* ctx;
        void* p[9] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
        explicit DeviceArrays(rt3_ctx* c) : ctx(c) {}
        ~DeviceArrays() { for (int k = 0; k < 9; k++) { rt3_buffer_free(ctx, p[k]); } }
        void* put(int slot, const void* host, size_t bytes, const char* what) {
            if (!host || bytes == 0) { return nullptr; }
            check(rt3_buffer_alloc(ctx, bytes, &p[slot]), what);
            return p[slot];
        }
    };
    for (size_t dev = 0; dev < 1 + this->helpers.size(); dev++) {
        rt3_ctx* c = dev == 0 ? this->ctx : this->helpers[dev - 1];
        DeviceArrays a(c);
        rt3_scene d = scene;
        d.faces = (const rt3_face*) a.put(0, scene.faces, (size_t) scene.n_faces * sizeof(rt3_face), "Could not allocate the device faces");
        d.vertices = (const rt3_vertex*) a.put(1, scene.vertices, (size_t) scene.n_vertices * sizeof(rt3_vertex), "Could not allocate the device vertices");
        for (size_t k = 0; k < host_ranges.size(); k++) {
            const Range& r = host_ranges[k];
            check(rt3_buffer_write(c, (rt3_face*) d.faces + r.first_face, scene.faces + r.first_face, r.n_faces * sizeof(rt3_face)), "Could not copy faces to the device");
            check(rt3_buffer_write(c, (rt3_vertex*) d.vertices + r.first_vertex, scene.vertices + r.first_vertex, r.n_vertices * sizeof(rt3_vertex)), "Could not copy vertices to the device");
        }
        for (size_t k = 0; k < deferred.size(); k++) {
            check(rt3_tessellate_spheres_device(c, &deferred[k].d, 1, deferred[k].first_vertex, deferred[k].first_face, (rt3_face*) d.faces, (rt3_vertex*) d.vertices, nullptr),
                  "Could not tessellate a sphere on the device");
        }
        const struct { int slot; const void** view; const void* host; size_t bytes; } small[] = {
            { 2, (const void**) &d.face_entity, scene.face_entity, (size_t) scene.n_faces * 4 }, { 3, (const void**) &d.face_material, scene.face_material, (size_t) scene.n_faces * 4 },
            { 4, (const void**) &d.spheres, scene.spheres, (size_t) scene.n_spheres * sizeof(rt3_sphere) }, { 5, (const void**) &d.sphere_color, scene.sphere_color, (size_t) scene.n_spheres * 12 },
            { 6, (const void**) &d.sphere_entity, scene.sphere_entity, (size_t) scene.n_spheres * 4 }, { 7, (const void**) &d.sphere_material, scene.sphere_material, (size_t) scene.n_spheres * 4 },
            { 8, (const void**) &d.materials, scene.materials, (size_t) scene.n_materials * sizeof(rt3_material) },
        };
        for (size_t k = 0; k < sizeof small / sizeof small[0]; k++) {
            *small[k].view = a.put(small[k].slot, small[k].host, small[k].bytes, "Could not allocate a device scene array");
            if (*small[k].view) { check(rt3_buffer_write(c, (void*) *small[k].view, small[k].host, small[k].bytes), "Could not copy a scene array to the device"); }
        }
        check(rt3_scene_upload_device(c, &d), dev == 0 ? "Could not build the scene on the device" : "Could not build the scene on a further device");
        if (dev == 0 && !deferred.empty()) {
            /* host copies for inspection (flat_faces / flat_vertices): what the kernels wrote */
            check(rt3_buffer_read(c, this->flat_faces.data(), d.faces, (size_t) scene.n_faces * sizeof(rt3_face)), "Could not read the faces back");
            check(rt3_buffer_read(c, this->flat_vertices.data(), d.vertices, (size_t) scene.n_vertices * sizeof(rt3_vertex)), "Could not read the vertices back");
        }
    }
}

void CudaRenderer::render(Camera& camera) const { this->render_samples(camera, 0, false); }

void CudaRenderer::render_progressive(Camera& camera, uint32_t passes, FrameCallback on_frame, void* user) const {
    if (this->settings.mode != RT3_MODE_PATHTRACE) { DLOG(fatal, "Progressive rendering needs the path-tracing mode."); }
    for (uint32_t pass = 0; pass < passes; pass++) {
        this->render_samples(camera, pass * this->settings.spp, pass > 0);
        if (on_frame) { on_frame(pass, camera.get_frame(), user); }
    }
}

namespace {
    rt3_camera camera_of(const Camera& camera) {
        rt3_camera cam;
        std::memset(&cam, 0, sizeof cam);
        const glm::vec3* src[4] = { &camera.origin, &camera.horizontal, &camera.vertical, &camera.lower_left_corner };
        float* dst[4] = { cam.origin, cam.horizontal, cam.vertical, cam.lower_left_corner };
        for (int i = 0; i < 4; i++) { dst[i][0] = src[i]->x; dst[i][1] = src[i]->y; dst[i][2] = src[i]->z; }
#ifdef RT3_HOST_CAMERA_CAMERA_HPP /* the thin lens exists only in this repo's Camera, not in the reference's */
        cam.lens_radius = camera.lens_radius;
        cam.lens_u[0] = camera.lens_u.x; cam.lens_u[1] = camera.lens_u.y; cam.lens_u[2] = camera.lens_u.z;
        cam.lens_v[0] = camera.lens_v.x; cam.lens_v[1] = camera.lens_v.y; cam.lens_v[2] = camera.lens_v.z;
#endif
        return cam;
    }

    /* A Portable Float Map of `channels` (3: "PF", 1: "Pf") floats per pixel, little-endian, rows bottom to top. */
    void write_pfm(const std::string& path, uint32_t width, uint32_t height, uint32_t channels, const float* data) {
        FILE* f = std::fopen(path.c_str(), "wb");
        if (!f) { DLOG(fatal, "Could not open '" + path + "' for writing."); }
        std::fprintf(f, "%s\n%u %u\n-1.0\n", channels == 3 ? "PF" : "Pf", width, height); /* negative scale: little-endian */
        const size_t row = (size_t) width * channels;
        bool ok = true;
        for (uint32_t y = height; y-- > 0 && ok;) { ok = std::fwrite(data + (size_t) y * row, sizeof(float), row, f) == row; }
        ok = (std::fclose(f) == 0) && ok;
        if (!ok) { DLOG(fatal, "Could not write '" + path + "'."); }
    }

    /* `params` for context i of n: the frame's row tiles are dealt round-robin over the contexts, within this process's own part
     * of a larger split (tile % (outer n) == i outer + p  implies  tile % outer == p). */
    rt3_params context_part(const rt3_params& params, uint32_t i, uint32_t n) {
        const uint32_t outer = params.part_count ? params.part_count : 1;
        rt3_params mine = params;
        mine.part_count = outer * n;
        mine.part_index = i * outer + params.part_index;
        return mine;
    }

    /* Adds one context's statistics to a total: counts add up; times are the longest one when the contexts ran concurrently,
     * their sum when they ran one after the other. */
    void add_stats(rt3_stats& total, const rt3_stats& st, bool concurrent) {
        total.rays += st.rays; total.sphere_tests += st.sphere_tests; total.face_tests += st.face_tests;
        total.accel_node_visits += st.accel_node_visits; total.accel_prim_tests += st.accel_prim_tests;
        total.beam_rays += st.beam_rays; total.beam_tests += st.beam_tests;
        total.rows_rendered += st.rows_rendered; total.kernel_launches += st.kernel_launches;
        if (concurrent) {
            if (st.device_ms > total.device_ms) { total.device_ms = st.device_ms; }
            if (st.trace_kernel_ms > total.trace_kernel_ms) { total.trace_kernel_ms = st.trace_kernel_ms; }
        } else {
            total.device_ms += st.device_ms; total.trace_kernel_ms += st.trace_kernel_ms;
        }
    }
}

rt3_params CudaRenderer::make_params(const Camera& camera, uint32_t first_sample, bool accumulate) const {
    rt3_params params;
    std::memset(&params, 0, sizeof params);
    params.width = camera.w();
    params.height = camera.h();
    params.mode = this->settings.mode;
    params.spp = this->settings.spp;
    params.max_depth = this->settings.max_depth;
    params.seed = this->settings.seed;
    params.flags = this->settings.flags | (accumulate ? RT3_FLAG_ACCUMULATE : 0u);
    if (this->flat_faces.size() + this->flat_spheres.size() > (size_t) this->settings.bvh_above) { params.flags |= RT3_FLAG_BVH; }
    params.first_sample = first_sample;
    params.tile_rows = this->settings.tile_rows;
    params.part_index = this->settings.part_index;
    params.part_count = this->settings.part_count;
    return params;
}

void CudaRenderer::render_samples(Camera& camera, uint32_t first_sample, bool accumulate) const {
    const rt3_camera cam = camera_of(camera);
    const rt3_params params = this->make_params(camera, first_sample, accumulate);
    if (this->helpers.empty()) {
        check(rt3_render(this->ctx, &cam, &params, camera.get_frame().d()), "Render failed");
        check(rt3_get_stats(this->ctx, &this->last_stats), "Could not read render statistics");
        return;
    }

    /* several devices: every context renders its tiles into the first device's frame (stores over NVLink), asynchronously;
     * the statistics calls below wait for each of them, then the frame is read once */
    const uint64_t n_pixels = (uint64_t) params.width * params.height;
    if (this->shared_pixels != n_pixels) {
        if (this->shared_frame) { check(rt3_frame_free(this->ctx, this->shared_frame), "Could not free the shared frame"); this->shared_frame = nullptr; this->shared_pixels = 0; }
        check(rt3_frame_alloc(this->ctx, n_pixels, &this->shared_frame), "Could not allocate the shared frame");
        this->shared_pixels = n_pixels;
    }
    const uint32_t n = (uint32_t) this->n_devices();
    for (uint32_t i = 0; i < n; i++) {
        const rt3_params mine = context_part(params, i, n);
        check(rt3_render_device(i == 0 ? this->ctx : this->helpers[i - 1], &cam, &mine, this->shared_frame, nullptr), "Render failed");
    }
    rt3_stats total;
    std::memset(&total, 0, sizeof total);
    for (uint32_t i = 0; i < n; i++) {
        rt3_stats st;
        check(rt3_get_stats(i == 0 ? this->ctx : this->helpers[i - 1], &st), "Could not read render statistics");
        if (i == 0) { total = st; } else { add_stats(total, st, true); }
    }
    check(rt3_frame_read(this->ctx, this->shared_frame, camera.get_frame().d(), n_pixels), "Could not read the frame");
    this->last_stats = total;
}

void CudaRenderer::read_radiance(uint32_t width, uint32_t height, std::vector<float>& rgb) const {
    const size_t n = (size_t) width * height * 3;
    rgb.assign(n, 0.0f);
    check(rt3_read_radiance(this->ctx, rgb.data(), width, height), "Could not read the radiance");
    if (this->helpers.empty()) { return; }
    /* every context returns zeros outside the rows it rendered: the frame is their sum */
    std::vector<float> part(n);
    for (size_t i = 0; i < this->helpers.size(); i++) {
        check(rt3_read_radiance(this->helpers[i], part.data(), width, height), "Could not read the radiance of a further device");
        for (size_t k = 0; k < n; k++) { rgb[k] += part[k]; }
    }
}

void CudaRenderer::write_radiance_pfm(uint32_t width, uint32_t height, const std::string& path) const {
    std::vector<float> rgb;
    this->read_radiance(width, height, rgb);
    write_pfm(path, width, height, 3, rgb.data());
}

void CudaRenderer::render_path_aovs(const Camera& camera, CudaPathAovs& out) const {
    if (this->settings.mode != RT3_MODE_PATHTRACE) { DLOG(fatal, "Path-traced AOVs need the path-tracing mode."); }
    const rt3_camera cam = camera_of(camera);
    rt3_params params = this->make_params(camera, 0, false);
    if (this->settings.aov_spp) { params.spp = this->settings.aov_spp; }
    const size_t n = (size_t) params.width * params.height;
    out.width = params.width; out.height = params.height;
    out.hit_prim.assign(n, 0u); out.hit_entity.assign(n, 0u); out.hit_t.assign(n, 0.0f); out.albedo.assign(3 * n, 0.0f); out.normal.assign(3 * n, 0.0f);
    const rt3_path_aovs dst = { out.hit_prim.data(), out.hit_entity.data(), out.hit_t.data(), out.albedo.data(), out.normal.data() };
    /* one context after the other, each writing its row tiles (the call is blocking) */
    const uint32_t n_ctx = (uint32_t) this->n_devices();
    rt3_stats total;
    std::memset(&total, 0, sizeof total);
    for (uint32_t i = 0; i < n_ctx; i++) {
        rt3_ctx* c = i == 0 ? this->ctx : this->helpers[i - 1];
        const rt3_params mine = context_part(params, i, n_ctx);
        check(rt3_render_path_aovs(c, &cam, &mine, &dst), "Path-traced AOVs failed");
        rt3_stats st;
        check(rt3_get_stats(c, &st), "Could not read render statistics");
        if (i == 0) { total = st; } else { add_stats(total, st, false); }
    }
    this->last_stats = total;
}

namespace {
    /* The filter's parameters for `camera`'s frame. Denoising needs a renderer on one device: with several, each context
     * holds only its own rows of the frame, and the filter reaches across them. `what` names the call in the refusal. */
    rt3_denoise_params denoise_params_of(const CudaDenoiseSettings& settings, const Camera& camera, size_t n_devices, const char* what) {
        if (n_devices > 1) {
            DLOG(fatal, std::string(what) + " needs a renderer on one device: with " + std::to_string(n_devices) +
                        " each context holds only its own rows of the frame, and the filter reaches across them.");
        }
        rt3_denoise_params params;
        std::memset(&params, 0, sizeof params);
        params.width = camera.w(); params.height = camera.h();
        params.iterations = settings.iterations;
        params.sigma_luminance = settings.sigma_luminance; params.sigma_normal = settings.sigma_normal; params.sigma_depth = settings.sigma_depth;
        return params;
    }
}

void CudaRenderer::denoise(Camera& camera, const CudaDenoiseSettings& settings, std::vector<float>* rgb) const {
    const rt3_denoise_params params = denoise_params_of(settings, camera, this->n_devices(), "Denoising");
    if (rgb) { rgb->assign((size_t) params.width * params.height * 3, 0.0f); }
    check(rt3_denoise(this->ctx, &params, camera.get_frame().d(), rgb ? rgb->data() : nullptr), "Denoising failed");
    check(rt3_get_stats(this->ctx, &this->last_stats), "Could not read the statistics");
}

void CudaRenderer::denoise_temporal(Camera& camera, const CudaDenoiseTemporalSettings& settings, bool reset, std::vector<float>* rgb) const {
    rt3_denoise_temporal_params params;
    std::memset(&params, 0, sizeof params);
    params.filter = denoise_params_of(settings.filter, camera, this->n_devices(), "Temporal denoising");
    params.alpha_color = settings.alpha_color; params.alpha_moments = settings.alpha_moments;
    params.depth_tolerance = settings.depth_tolerance; params.normal_cos = settings.normal_cos;
    params.reset = reset ? 1u : 0u;
    if (rgb) { rgb->assign((size_t) params.filter.width * params.filter.height * 3, 0.0f); }
    check(rt3_denoise_temporal(this->ctx, &params, camera.get_frame().d(), rgb ? rgb->data() : nullptr, nullptr), "Temporal denoising failed");
    check(rt3_get_stats(this->ctx, &this->last_stats), "Could not read the statistics");
}

void CudaRenderer::write_path_aovs_pfm(const CudaPathAovs& aovs, const std::string& dir) const {
    const std::string base = dir.empty() ? std::string(".") : dir;
    write_pfm(base + "/albedo.pfm", aovs.width, aovs.height, 3, aovs.albedo.data());
    write_pfm(base + "/normal.pfm", aovs.width, aovs.height, 3, aovs.normal.data());
    write_pfm(base + "/depth.pfm", aovs.width, aovs.height, 1, aovs.hit_t.data());
}

/* Factory of this backend (reference Renderer.hpp:63; counterpart of SequentialRenderer.cpp:315-323). */
Renderer* RayTracer::initialize_renderer() {
    int device = 0;
    CudaRenderSettings settings = CudaRenderSettings::from_environment(&device);
    const std::vector<int> devices = CudaRenderSettings::devices_from_environment();
    CudaRenderer* renderer = devices.size() > 1 ? new CudaRenderer(devices) : new CudaRenderer(devices[0]);
    renderer->set_settings(settings);
    return (Renderer*) renderer;
}
