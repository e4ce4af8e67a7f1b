/* renderer/CudaRenderer.hpp — the B200 backend behind RayTracer::Renderer.
 *
 * Replaces SequentialRenderer / VulkanRenderer (reference
 * src/lib/renderer/SequentialRenderer.hpp:25-45, VulkanRenderer.hpp:40-95) for
 * the render path: prerender() flattens the ECS entities exactly as the
 * reference does (SequentialRenderer.cpp:174-266) and uploads them once;
 * render() runs the CUDA core through the C ABI of include/rt3cuda.h and writes
 * Camera::get_frame() in place. Failures go through DLOG(fatal, ...) like the
 * reference's backends.
 *
 * Written against the reference's own header names (renderer/Renderer.hpp,
 * entities/..., camera/Camera.hpp, tools/Array.hpp), so the same source
 * builds standalone against raytracer-3_b200/host/ and inside the reference
 * tree (INTEGRATION.md; oracle/Makefile target `dropin`).
 */
#ifndef RT3_HOST_RENDERER_CUDA_RENDERER_HPP
#define RT3_HOST_RENDERER_CUDA_RENDERER_HPP

#include <cstdint>
#include <map>
#include <string>
#include <vector>

#include "renderer/Renderer.hpp"
#include "rt3cuda.h"

namespace RayTracer {
    /* Material of an entity for the bounce loop. The reference's entities only carry a colour
     * (Sphere.hpp:44 etc.), so materials are a side table keyed by entity index. */
    struct Material {
        enum Kind { lambertian = RT3_MAT_LAMBERTIAN, metal = RT3_MAT_METAL, dielectric = RT3_MAT_DIELECTRIC };
        Kind kind = lambertian;
        glm::vec3 albedo = glm::vec3(0.5f, 0.5f, 0.5f);
        float fuzz = 0.0f;
        float ior = 1.5f;
    };

    struct CudaRenderSettings {
        uint32_t mode = RT3_MODE_REFERENCE; /* RT3_MODE_REFERENCE reproduces the reference's image */
        uint32_t spp = 100;
        uint32_t max_depth = 50;
        uint32_t seed = 1;
        uint32_t flags = 0;
        /* Closest hits through the device-built hierarchy (RT3_FLAG_BVH) when the scene has more primitives than this;
         * the brute-force sweep below it. The two give identical frames (DESIGN.md 3.5), so this is purely a matter of speed:
         * the sweep wins while its records stay in the constant cache. 0 = always the hierarchy, UINT32_MAX = never. */
        uint32_t bvh_above = 768;
        bool analytic_spheres = false;      /* keep ECS spheres analytic instead of tessellating them */
        bool device_tessellation = false;   /* build the flattened scene in device memory: ECS spheres are tessellated there (rt3_tessellate_spheres_device),
                                             * the host's triangles / object files are copied next to them, and nothing is derived on the host (rt3_scene_upload_device) */
        uint32_t tile_rows = 8, part_index = 0, part_count = 1;
        uint32_t aov_spp = 0; /* samples per pixel of render_path_aovs; 0: spp */
        /* Reads RT3_MODE (reference|pathtrace), RT3_SPP, RT3_DEPTH, RT3_SEED, RT3_ANALYTIC_SPHERES, RT3_DEVICE_TESSELLATION, RT3_BVH, RT3_BVH_ABOVE, RT3_DEVICE. */
        static CudaRenderSettings from_environment(int* device);
        /* RT3_DEVICES = comma-separated device ids ("0,1,2,3") or "all"; falls back to the single RT3_DEVICE. */
        static std::vector<int> devices_from_environment();
    };

    /* AOVs of a path-traced frame (rt3_render_path_aovs): width * height pixels in frame order, albedo and normal 3 floats each. */
    struct CudaPathAovs {
        uint32_t width = 0, height = 0;
        std::vector<uint32_t> hit_prim, hit_entity;
        std::vector<float> hit_t, albedo, normal;
    };

    /* Parameters of CudaRenderer::denoise (rt3_denoise_params; SVGF's defaults). */
    struct CudaDenoiseSettings {
        uint32_t iterations = 5;
        float sigma_luminance = 4.0f, sigma_normal = 128.0f, sigma_depth = 1.0f;
    };

    /* Parameters of CudaRenderer::denoise_temporal (rt3_denoise_temporal_params; SVGF's defaults). */
    struct CudaDenoiseTemporalSettings {
        CudaDenoiseSettings filter;
        float alpha_color = 0.2f, alpha_moments = 0.2f, depth_tolerance = 0.05f, normal_cos = 0.9f;
    };

    class CudaRenderer : public Renderer {
        rt3_ctx* ctx;                 /* first device: owns the frame when there are several */
        std::vector<rt3_ctx*> helpers; /* further devices (SURVEY 8e): each renders its row tiles straight into ctx's frame */
        mutable uint32_t* shared_frame;
        mutable uint64_t shared_pixels;
        CudaRenderSettings settings;
        std::map<size_t, Material> materials;
        mutable rt3_stats last_stats;
        void render_samples(Camera& camera, uint32_t first_sample, bool accumulate) const;
        rt3_params make_params(const Camera& camera, uint32_t first_sample, bool accumulate) const;
        void release() noexcept;

    public:
        explicit CudaRenderer(int device = 0);
        /* One context per listed device; a frame is split in row tiles of settings.tile_rows rows dealt round-robin over
         * them, the scene is replicated. The result is the one-device frame bit for bit (global pixel indices seed the RNG). */
        explicit CudaRenderer(const std::vector<int>& devices);
        size_t n_devices() const { return 1 + this->helpers.size(); }
        CudaRenderer(const CudaRenderer&) = delete;
        virtual ~CudaRenderer();

        void set_settings(const CudaRenderSettings& s) { this->settings = s; }
        const CudaRenderSettings& get_settings() const { return this->settings; }
        /* Applies to the next prerender(). */
        void set_material(size_t entity_index, const Material& material) { this->materials[entity_index] = material; }
        void clear_materials() { this->materials.clear(); }

        virtual void prerender(const Tools::Array<ECS::RenderEntity*>& entities);
        virtual void render(Camera& camera) const;

        /* Online / progressive mode (the headless counterpart of the reference's VulkanOnlineRenderer frame loop,
         * VulkanOnlineRenderer.cpp:637-735): `passes` renders of settings.spp samples each into the same accumulators
         * (RT3_FLAG_ACCUMULATE); after every pass the camera's frame holds the image over all samples so far and
         * `on_frame(pass, camera.get_frame())` is called if given. The last frame equals one render() of
         * passes * spp samples bit for bit. Path tracing only. */
        typedef void (*FrameCallback)(uint32_t pass, const Frame& frame, void* user);
        void render_progressive(Camera& camera, uint32_t passes, FrameCallback on_frame = nullptr, void* user = nullptr) const;

        /* Float AOV of the last path-traced render(): mean linear radiance (before gamma and the 8-bit pack), 3 floats per
         * pixel in frame order (rt3_read_radiance; with several devices each context contributes the rows it rendered). */
        void read_radiance(uint32_t width, uint32_t height, std::vector<float>& rgb) const;
        /* The same as a Portable Float Map ("PF", little-endian, rows bottom to top), the float counterpart of Frame::to_ppm. */
        void write_radiance_pfm(uint32_t width, uint32_t height, const std::string& path) const;

        /* AOVs of the path tracer's primary rays for the frame render() would path-trace with these settings (its first
         * settings.aov_spp samples, or spp): the albedo and normal buffers an image denoiser takes next to the noisy colour,
         * and per pixel the primitive, entity and distance of the first sample's hit. With several devices every context
         * renders its row tiles into the same arrays. Leaves the accumulators of render() / render_progressive() alone. */
        void render_path_aovs(const Camera& camera, CudaPathAovs& out) const;
        /* Denoises the last render() / render_progressive() of this camera's frame (rt3_denoise), guided by the last
         * render_path_aovs() with the same camera, and writes the result into the camera's frame; `rgb`, when given, receives
         * the linear float image (3 per pixel). One device only: each context of a renderer with several holds only its own
         * rows, and the filter reaches across them. */
        void denoise(Camera& camera, const CudaDenoiseSettings& settings = {}, std::vector<float>* rgb = nullptr) const;
        /* denoise() with the history of the earlier calls reprojected through the camera's motion and accumulated
         * (rt3_denoise_temporal; `reset` drops the history first). Render each frame with its own seed. One device only. */
        void denoise_temporal(Camera& camera, const CudaDenoiseTemporalSettings& settings = {}, bool reset = false, std::vector<float>* rgb = nullptr) const;
        /* albedo.pfm and normal.pfm ("PF", 3 channels) and depth.pfm ("Pf", hit_t; +inf where the primary ray missed) in `dir`. */
        void write_path_aovs_pfm(const CudaPathAovs& aovs, const std::string& dir) const;

        /* Device timings / ray counters of the last render(). */
        const rt3_stats& stats() const { return this->last_stats; }

        /* The flattened scene of the last prerender() (host copies, for inspection and tests). */
        std::vector<rt3_face> flat_faces;
        std::vector<rt3_vertex> flat_vertices;
        std::vector<uint32_t> flat_face_entity;
        std::vector<rt3_sphere> flat_spheres;
    };
}

#endif
