/* rt3cuda.h — C ABI of the B200-native render core (librt3cuda.so).
 *
 * This is the drop-in boundary for RayTracer-3's per-pixel hot path. A host
 * renderer backend (raytracer-3_b200/host/CudaRenderer.cpp, or a backend a
 * maintainer adds to the reference tree — see INTEGRATION.md) implements the
 * reference plug-in interface
 *     RayTracer::Renderer::prerender(const Tools::Array<ECS::RenderEntity*>&)
 *     RayTracer::Renderer::render(Camera&) const
 *     RayTracer::initialize_renderer()
 * (reference src/lib/renderer/Renderer.hpp:34-63) on top of these calls:
 *
 *   reference interface                                   this ABI
 *   ---------------------------------------------------   --------------------------
 *   initialize_renderer()        Renderer.hpp:63          rt3_create
 *   ~Renderer()                  Renderer.hpp:45          rt3_destroy
 *   Renderer::prerender upload   VulkanRenderer.cpp:266   rt3_scene_upload
 *   Renderer::render             Renderer.hpp:50,         rt3_render / rt3_render_aov
 *                                SequentialRenderer.cpp:269-308
 *   DLOG(fatal, msg)             Main.cpp:305-308         non-zero status + rt3_last_error
 *
 * Plain C: pointers and sizes only, no C++ or torch types, no exceptions across
 * the boundary. All functions return 0 on success, a negative rt3 status on
 * failure; rt3_last_error() then describes it (thread-local string).
 * There is no CPU fallback: without a CUDA device rt3_create fails.
 */
#ifndef RT3CUDA_H
#define RT3CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT3_OK 0
#define RT3_ERR_INVALID (-1)   /* bad argument / inconsistent scene */
#define RT3_ERR_CUDA (-2)      /* CUDA runtime error (message has the cudaError string) */
#define RT3_ERR_NO_SCENE (-3)  /* render called before rt3_scene_upload */
#define RT3_ERR_NO_DEVICE (-4) /* no usable CUDA device */

/* ---- scene -------------------------------------------------------------- */

/* The reference's flattened face record, byte for byte
 * (GFace, reference src/lib/renderer/Vertex.hpp:39-51; sizeof == 48). */
typedef struct rt3_face {
    uint32_t v1, v2, v3; /* indices into the vertex array */
    uint32_t _pad0;
    float normal[3];     /* host-computed face normal (Triangle.cpp:48, Object.cpp:193, Sphere.cpp:153) */
    float _pad1;
    float color[3];      /* baked flat colour (Sphere.cpp:155, Object.cpp:194) / albedo */
    float _pad2;
} rt3_face;

/* The reference's vertex record (glm::vec4, w = 0; SequentialRenderer.hpp:31). */
typedef struct rt3_vertex {
    float x, y, z, w;
} rt3_vertex;

#define RT3_MAT_LAMBERTIAN 0u
#define RT3_MAT_METAL 1u
#define RT3_MAT_DIELECTRIC 2u

/* Material record. The reference ECS carries only a colour per entity
 * (Sphere.hpp:44, Triangle.hpp:34, Object.hpp:37); the material table is the
 * extension the bounce loop needs (raytracer_v4.glsl:255-283 reserves
 * obj_material for it). */
typedef struct rt3_material {
    uint32_t kind;   /* RT3_MAT_* */
    float albedo[3]; /* attenuation for Lambertian / metal; ignored for dielectric */
    float fuzz;      /* metal: radius of the perturbation ball, clamped to [0,1] */
    float ior;       /* dielectric: index of refraction */
    float _pad[2];
} rt3_material;

/* Analytic sphere (raytracer_v4.glsl:43-50 `Sphere`): centre + radius.
 * A negative radius gives the hollow-glass inward-normal sphere. */
typedef struct rt3_sphere {
    float cx, cy, cz, r;
} rt3_sphere;

/* Everything is copied during rt3_scene_upload; the caller keeps ownership
 * (the reference deletes its entities right after render, Main.cpp:286-288).
 * Primitive ids in AOVs: faces are 0..n_faces-1 in array order (the reference's
 * order, SequentialRenderer.cpp:174-195), spheres follow at n_faces + i
 * (faces are tested before spheres, raytracer_v4.glsl:227-245). */
typedef struct rt3_scene {
    uint32_t n_faces;
    uint32_t n_vertices;
    const rt3_face* faces;
    const rt3_vertex* vertices;
    const uint32_t* face_material; /* per face index into materials; NULL: Lambertian(face colour) */
    const uint32_t* face_entity;   /* per face entity id; NULL: 0 */

    uint32_t n_spheres;
    uint32_t n_materials;
    const rt3_sphere* spheres;
    const float* sphere_color;       /* 3 floats per sphere: flat colour in reference mode, albedo when sphere_material is NULL */
    const uint32_t* sphere_material; /* per sphere index into materials; NULL: Lambertian(sphere colour) */
    const uint32_t* sphere_entity;   /* per sphere entity id; NULL: 0 */
    const rt3_material* materials;
} rt3_scene;

/* UV sphere to be tessellated (the fields of ECS::Sphere, reference src/lib/entities/Sphere.hpp:33-45). */
typedef struct rt3_uv_sphere {
    float center[3];
    float radius;
    uint32_t n_meridians; /* >= 1 */
    uint32_t n_parallels; /* >= 3 (Sphere.cpp:101) */
    float color[3];
    uint32_t entity;      /* entity id recorded for its faces */
} rt3_uv_sphere;

/* ---- camera ------------------------------------------------------------- */

/* The four public vectors of the reference Camera (camera/Camera.hpp:27-34;
 * GPU mirror GCameraData, VulkanRenderer.hpp:32-37), plus an optional thin
 * lens (lens_radius == 0: pinhole, lens_u / lens_v ignored). */
typedef struct rt3_camera {
    float origin[3];
    float horizontal[3];
    float vertical[3];
    float lower_left_corner[3];
    float lens_radius;
    float lens_u[3];
    float lens_v[3];
} rt3_camera;

/* ---- render parameters -------------------------------------------------- */

/* RT3_MODE_REFERENCE: the reference's ray caster, in the reference's
 *   arithmetic order with no FMA contraction: one un-jittered primary ray per
 *   pixel, brute-force closest hit, flat baked colour or sky gradient
 *   (SequentialRenderer.cpp:47-109,284-297). spp/max_depth/seed are ignored.
 *   All rows are rendered (the reference's CPU loop skips the last row,
 *   SequentialRenderer.cpp:286; its GLSL renders it, raytracer_v3.glsl:193).
 * RT3_MODE_PATHTRACE: spp jittered samples per pixel, multi-bounce
 *   Lambertian / metal / dielectric shading up to max_depth segments,
 *   order-independent fixed-point accumulation, gamma-2 resolve. */
#define RT3_MODE_REFERENCE 0u
#define RT3_MODE_PATHTRACE 1u

#define RT3_FLAG_NO_JITTER 0x1u /* pathtrace: sample pixel centres (deterministic primary rays) */
#define RT3_FLAG_NO_GAMMA 0x2u  /* pathtrace: resolve the linear mean instead of its square root */
#define RT3_FLAG_ACCUMULATE 0x8u /* pathtrace, progressive refinement: keep the accumulators of the previous render of this context
                                 * and add this call's samples [first_sample, first_sample + spp) to them; the frame is resolved
                                 * over first_sample + spp samples. k calls of n spp produce exactly the frame of one call of
                                 * k*n spp (integer accumulation). Checked (RT3_ERR_INVALID otherwise): same scene upload, frame
                                 * size, partition, seed, max_depth and sampling flags as the accumulated render, and
                                 * first_sample == the end of the range accumulated so far. */
#define RT3_FLAG_UNIFORM_SKY 0x10u /* pathtrace: a miss returns radiance (1, 1, 1) instead of the reference's sky gradient
                                 * (SequentialRenderer.cpp:105-107): the white-furnace configuration the energy-conservation
                                 * tests use (an albedo-1 scene must resolve to exactly white) */
#define RT3_FLAG_BVH 0x4u       /* closest hits through a bounding-volume hierarchy built on the device at the first such render
                                 * after rt3_scene_upload, instead of the reference's brute-force loop over every primitive
                                 * (SequentialRenderer.cpp:55-95). The frame and the AOVs are identical, bit for bit. */

typedef struct rt3_params {
    uint32_t width;
    uint32_t height;
    uint32_t mode;      /* RT3_MODE_* */
    uint32_t spp;       /* samples per pixel (pathtrace), 1..65535 */
    uint32_t max_depth; /* maximum ray segments per path (pathtrace), >= 1 */
    uint32_t seed;
    uint32_t flags;     /* RT3_FLAG_* */
    /* Row-tile partition (multi-GPU): the image is cut into tiles of tile_rows
     * rows; this context renders tiles t with t % part_count == part_index.
     * part_count <= 1 renders everything. Results do not depend on the
     * partition (per-pixel RNG counters use the global pixel index). */
    uint32_t tile_rows;
    uint32_t part_index;
    uint32_t part_count;
    uint32_t first_sample; /* pathtrace: sample index of the first of this call's spp samples (0 for a one-shot render) */
} rt3_params;

/* Timings and counters of the most recent render on this context. */
typedef struct rt3_stats {
    double device_ms;       /* CUDA-event time of all render kernels (clear + trace + resolve), on the render stream */
    double trace_kernel_ms; /* CUDA-event time of the dominant kernel alone (reference_kernel / pathtrace_kernel) */
    double h2d_ms;          /* host->device copies of the most recent rt3_scene_upload on this context (a render copies nothing to the
                             * device: camera and parameters travel as kernel arguments); 0 after rt3_scene_upload_device */
    double d2h_ms;          /* device->host copy of the frame / AOVs */
    uint64_t rays;          /* ray segments traced (primary + bounce), counted by the kernel */
    uint64_t sphere_tests;  /* ray-sphere tests = rays * n_spheres (brute force) */
    uint64_t face_tests;    /* ray-triangle tests = rays * n_faces */
    uint32_t kernel_launches;
    uint32_t rows_rendered; /* rows owned by this partition */
    /* RT3_FLAG_BVH renders: sphere_tests / face_tests are 0 (no brute-force sweep) and these count the traversal */
    uint64_t accel_node_visits; /* hierarchy nodes read */
    uint64_t accel_prim_tests;  /* exact ray-primitive tests run in leaves */
    double accel_build_ms;      /* device time of the hierarchy build for the current scene */
    uint32_t accel;             /* 1 if the most recent render used the hierarchy */
    uint32_t accel_stack_overflows; /* subtrees the traversal could not stack (never, for trees this library builds: depth <= 94 of 128); a render
                                 * with a non-zero count fails (rt3_render) or makes rt3_get_stats fail (rt3_render_device) */
    /* the most recent scene upload on this context (the reference's prerender, Main.cpp:284) */
    double upload_ms;           /* wall clock of rt3_scene_upload / rt3_scene_upload_device, call to return */
    double upload_device_ms;    /* CUDA-event time of the kernels that derive bounds, boxes, prefilter records and the scene basis */
    /* pathtrace renders of resident sphere scenes through the sweep: primary rays are traced against a candidate list per chunk of path
     * items instead of sweeping the scene (same hits, bit for bit); sphere_tests counts what was really tested:
     * (rays - beam_rays) * n_spheres + beam_tests. Renders through the hierarchy (RT3_FLAG_BVH) do the same with the candidates a beam's
     * walk of the trees collected: those primary rays did not traverse (accel_node_visits includes the nodes the beams read) */
    uint64_t beam_rays;         /* primary rays traced against a candidate list */
    uint64_t beam_tests;        /* exact tests those rays ran (spheres; through the hierarchy: spheres and triangles) */
} rt3_stats;

typedef struct rt3_ctx rt3_ctx;

/* ---- entry points ------------------------------------------------------- */

const char* rt3_last_error(void);

/* Creates a context on CUDA device `device` (>= 0). */
int rt3_create(rt3_ctx** out, int device);
int rt3_destroy(rt3_ctx* ctx);

/* Flattens the scene into device SoA arrays (replacing any previous scene): the input arrays are copied to the device as
 * they are and everything derived from them (exact-test arrays, bounding spheres and boxes, prefilter records, the scene
 * basis) is built there by kernels; the host does no per-primitive work. Validation errors (a face index or a material
 * index out of range, an unknown material kind) are found on the device and reported here: the first one in input order. */
int rt3_scene_upload(rt3_ctx* ctx, const rt3_scene* scene);

/* The same for a scene that already lies in this context's device memory: every pointer of `scene` is a DEVICE pointer
 * (faces, vertices, spheres and materials 16-byte aligned), e.g. buffers from rt3_buffer_alloc filled by
 * rt3_tessellate_spheres_device and rt3_buffer_write. Nothing is copied from the host. The buffers are only read during
 * the call. (The reference keeps its flattened scene on the GPU the same way, VulkanRenderer.cpp:266-399.) */
int rt3_scene_upload_device(rt3_ctx* ctx, const rt3_scene* scene);

/* Plain device memory on the context's GPU for such scenes; write / read are blocking copies. */
int rt3_buffer_alloc(rt3_ctx* ctx, uint64_t bytes, void** device_ptr);
int rt3_buffer_free(rt3_ctx* ctx, void* device_ptr);
int rt3_buffer_write(rt3_ctx* ctx, void* device_dst, const void* host_src, uint64_t bytes);
int rt3_buffer_read(rt3_ctx* ctx, void* host_dst, const void* device_src, uint64_t bytes);

/* Renders into a HOST frame of width*height packed pixels, reference packing
 * r<<24 | g<<16 | b<<8 | 0xFF, index y*width + x, row 0 = top
 * (SequentialRenderer.cpp:297, Frame.hpp:44). With a partition, only the rows
 * this context owns are written. Blocking, like the reference's render(). */
int rt3_render(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, uint32_t* host_frame);

/* As rt3_render, and also returns per pixel the closest-hit AOVs of the
 * primary ray: primitive id (0xFFFFFFFF on a miss), entity id (0xFFFFFFFF on
 * a miss) and hit distance along the un-normalised primary direction (+inf on
 * a miss). Any of the three output pointers may be NULL.
 * Only RT3_MODE_REFERENCE is supported. */
int rt3_render_aov(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, uint32_t* host_frame,
                   uint32_t* host_hit_prim, uint32_t* host_hit_entity, float* host_hit_t);

/* AOVs of a path-traced render: the buffers an image denoiser takes next to the noisy colour (albedo, normal) and the
 * primary hit per pixel (primitive, entity, depth). Host pointers, width*height pixels in frame order; any may be NULL. */
typedef struct rt3_path_aovs {
    uint32_t* hit_prim;   /* primitive id of the closest hit of sample first_sample (0xFFFFFFFF on a miss) */
    uint32_t* hit_entity; /* its entity id (0xFFFFFFFF on a miss) */
    float* hit_t;         /* its distance along the UNIT primary direction (+inf on a miss); rt3_render_aov's hit_t is measured
                           * along the un-normalised reference-mode direction instead */
    float* albedo;        /* 3 per pixel, mean over the samples: the albedo the path tracer multiplies by at the first hit (the
                           * material's, or the primitive's colour without a material; 1 for a dielectric); a miss: the sky of
                           * that direction (1 under RT3_FLAG_UNIFORM_SKY) */
    float* normal;        /* 3 per pixel, mean over the samples (not renormalised) of the front-facing normal at the first hit
                           * (faces: the stored face normal; spheres: (hit point - centre) / radius); a miss: 0 */
} rt3_path_aovs;

/* Renders the AOVs of the path tracer's primary rays for RT3_MODE_PATHTRACE parameters: exactly the primary rays a render
 * with the same parameters traces for its samples [first_sample, first_sample + spp) of every owned pixel (seed, jitter,
 * thin lens, partition), with the path tracer's closest-hit tests. Reads spp (the number of AOV samples: the parameters
 * of a 500-spp render with spp = 16 give the AOVs of that render's first 16 samples), seed, first_sample, the partition
 * and the flags RT3_FLAG_NO_JITTER, RT3_FLAG_UNIFORM_SKY and RT3_FLAG_BVH; max_depth and the other flags are ignored.
 * Writes only the owned rows. Sums are kept in fixed point (2^24), so the result does not depend on scheduling,
 * partition or GPU count. Blocking. The path tracer's accumulators and RT3_FLAG_ACCUMULATE state are not touched:
 * rt3_read_radiance and a following accumulating render behave as if this call had not happened. rt3_get_stats then
 * describes this call (device_ms, trace_kernel_ms, rays = primary rays traced, the test or hierarchy counters). */
int rt3_render_path_aovs(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, const rt3_path_aovs* out);

/* Parameters of rt3_denoise (defaults: SVGF's, Schied et al. 2017). */
typedef struct rt3_denoise_params {
    uint32_t width, height; /* the frame host_frame and host_rgb hold: must be the render's */
    uint32_t iterations;   /* à-trous passes, 1..8 (default 5: steps 1, 2, 4, 8, 16, a reach of 64 pixels) */
    float sigma_luminance; /* luminance edge-stopping, finite and > 0 (default 4) */
    float sigma_normal;    /* exponent of the normal term, a whole number in 1..1024 (default 128) */
    float sigma_depth;     /* relative depth edge-stopping, finite and > 0 (default 1) */
} rt3_denoise_params;

/* Denoises the last path-traced render on this context: an edge-avoiding à-trous wavelet filter (the spatial filter of
 * SVGF) on its radiance (bit-equal to rt3_read_radiance), divided by the albedo and guided by the normal and depth of the
 * last rt3_render_path_aovs on this context; the result is multiplied by the albedo again and resolved like the render's
 * frame (gamma 2 unless the render had RT3_FLAG_NO_GAMMA, 8-bit pack). The formulas are in include/rt3_denoise.h and
 * DESIGN.md 3.8. Needs both calls to cover the whole frame (part_count <= 1) with the same width, height, camera and
 * scene upload; otherwise RT3_ERR_INVALID, with a message that names the condition, and nothing changes. Writes
 * width*height packed pixels to host_frame and 3 linear floats per pixel to host_rgb; either may be NULL. Blocking. The
 * accumulators, the AOV buffers and the RT3_FLAG_ACCUMULATE state are not touched. rt3_get_stats then describes this
 * call (device_ms, kernel_launches, rays = 0). */
int rt3_denoise(rt3_ctx* ctx, const rt3_denoise_params* params, uint32_t* host_frame, float* host_rgb);

/* Parameters of rt3_denoise_temporal (defaults: SVGF's). */
typedef struct rt3_denoise_temporal_params {
    rt3_denoise_params filter; /* the spatial passes, checked exactly as rt3_denoise checks them */
    float alpha_color;         /* (0, 1], default 0.2: smallest weight of the new frame in the colour history */
    float alpha_moments;       /* (0, 1], default 0.2: the same for the luminance moments */
    float depth_tolerance;     /* finite, > 0, default 0.05: relative depth test of a history tap */
    float normal_cos;          /* [-1, 1], default 0.9: smallest n^_p . n^_q of a history tap */
    uint32_t reset;            /* nonzero: ignore and replace the context's history */
} rt3_denoise_temporal_params;

/* rt3_denoise with temporal accumulation (the temporal half of SVGF): for a sequence of frames of one scene upload and
 * size whose camera moves, each pixel's surface point (the primary ray of sample first_sample of the last
 * rt3_render_path_aovs, at its depth; a miss: its direction) is reprojected into the previous call's camera, the 2x2
 * bilinear taps of the history there that agree in geometry (both misses, or both hits within depth_tolerance of the
 * distance and normal_cos of the normal) are blended into an exponential moving average of the demodulated colour and
 * of the luminance moments, and the luminance variance comes from those moments once 4 frames are behind a pixel. The
 * unchanged à-trous passes of rt3_denoise then filter the accumulated colour. Formulas: include/rt3_denoise.h, DESIGN.md
 * 3.9. Takes and checks what rt3_denoise takes and checks (messages name rt3_denoise_temporal), plus the parameters
 * above. The history (unfiltered colour, moments and length per pixel, the guide, and the camera, size and scene upload
 * that produced it) lives on the context; it is dropped, and every pixel starts at length 1, when reset is set, when
 * there is none yet, or when the width, height or scene upload differ from the history's. Render every frame with its
 * own seed: repeated noise is not averaged away. A call with no usable history anywhere is bit-equal to rt3_denoise.
 * Writes host_frame and host_rgb as rt3_denoise does, and each pixel's new history length to host_history_length; any
 * may be NULL. Blocking. A refused call (RT3_ERR_INVALID) changes nothing; a call that fails with a CUDA error drops the
 * history. The accumulators, the AOV buffers and the RT3_FLAG_ACCUMULATE state are not touched, and rt3_denoise is not
 * affected by it. rt3_get_stats then describes this call (device_ms, kernel_launches, rays = 0). The history is the one
 * rt3_denoise_staged_temporal uses on this context. */
int rt3_denoise_temporal(rt3_ctx* ctx, const rt3_denoise_temporal_params* params, uint32_t* host_frame, float* host_rgb,
                         float* host_history_length);

/* Denoising a frame rendered in parts (several contexts, GPUs or processes, each with its own row tiles): every part
 * prepares its own rows into one shared stage buffer (rt3_denoise_stage), and the stage's owner filters the whole frame
 * from it (rt3_denoise_staged). The result is bit-equal to rt3_denoise of a one-context render of the same frame: every
 * input of the filter's prepare step is per pixel and does not depend on the partition.
 *
 * The stage is plain device memory of rt3_denoise_stage_words(width, height) 32-bit words from rt3_frame_alloc(owner, ...),
 * shared like a frame (rt3_frame_export / rt3_frame_import / rt3_frame_attach / rt3_frame_release). Layout, n = width *
 * height pixels in frame order (index y * width + x), offsets in words:
 *   [0, 4n)           colour plane: rt3_dn_px per pixel (16 B: radiance / max(albedo, 1e-3) per channel, its luminance);
 *   [4n, 8n)          guide plane:  rt3_dn_guide per pixel (16 B: unit normal, depth);
 *   [8n, 11n)         albedo plane: 3 floats per pixel, the AOV albedo as it is;
 *   [F, F + 2 height) one 64-bit fingerprint per row (little-endian), F = 11n rounded up to an even word.
 * A row's fingerprint is a nonzero hash of the caller's frame_tag and of everything that changes the filter's input
 * pixels: width, height, the camera, seed, max_depth, the accumulated sample range and resolve count, RT3_FLAG_NO_JITTER,
 * RT3_FLAG_UNIFORM_SKY, RT3_FLAG_NO_GAMMA, tile_rows, part_count, and the AOV call's seed, spp, first_sample and sampling
 * flags (not RT3_FLAG_BVH or part_index: they change no pixel). rt3_frame_alloc zeroes the stage, so a row no part
 * staged has fingerprint 0. */

/* Words (uint32) of the stage for a width x height frame; 0 for an empty frame or when it would exceed what
 * rt3_frame_alloc takes (2^32 - 1 words). */
uint64_t rt3_denoise_stage_words(uint32_t width, uint32_t height);

/* This context's part of a frame rendered in parts: prepares the rows its last path-traced render owns (the radiance
 * divided by the albedo, the luminance, the guide and the raw albedo) and stores them and one fingerprint per owned row
 * into device_stage, which uses full-frame indexing and may be a peer or IPC mapping. Checks what rt3_denoise checks,
 * except that a partition is allowed: the render and the AOVs must have the same one (tile_rows, part_index,
 * part_count). device_stage must not be NULL. A refusal is RT3_ERR_INVALID with a message that names the condition,
 * and nothing changes. Asynchronous on cuda_stream (a cudaStream_t); NULL means the stream of the render that filled the
 * accumulators. rt3_get_stats then waits for it and describes it (device_ms, kernel_launches = 1, rows_rendered). The
 * accumulators, the AOV buffers and the RT3_FLAG_ACCUMULATE state are not touched. */
int rt3_denoise_stage(rt3_ctx* ctx, const rt3_denoise_params* params, uint64_t frame_tag, uint32_t* device_stage, void* cuda_stream);

/* On the stage's owner, which must be one of the parts, after every part's rt3_denoise_stage has completed: computes the
 * fingerprint from its own render and AOV state (checked as by rt3_denoise_stage), compares it with every row's, and
 * refuses (RT3_ERR_INVALID, naming the first row that differs and how many do; nothing written) when a row was not
 * staged for this frame: a part that did not run, a stale row of an earlier frame_tag, or a part with other parameters.
 * Then filters the whole frame from the stage with rt3_denoise's kernels and writes host_frame and host_rgb as
 * rt3_denoise does (the gamma follows this context's render). Blocking. The accumulators, the AOV buffers and the
 * RT3_FLAG_ACCUMULATE state are not touched; rt3_get_stats then describes this call (device_ms of the filter). */
int rt3_denoise_staged(rt3_ctx* ctx, const rt3_denoise_params* params, uint64_t frame_tag, const uint32_t* device_stage,
                       uint32_t* host_frame, float* host_rgb);

/* rt3_denoise_staged with temporal accumulation: the counterpart of rt3_denoise_temporal for a frame rendered in parts.
 * On the stage's owner, after every part's rt3_denoise_stage for frame_tag has completed (the parts stage exactly as for
 * rt3_denoise_staged and hold no history). Checks and refuses what rt3_denoise_staged does (NULL device_stage, a frame
 * too large for a stage, every row whose fingerprint differs from the owner's, naming the first and the count), plus
 * NULL params and the temporal parameters as rt3_denoise_temporal checks them; messages name
 * rt3_denoise_staged_temporal. Each pixel's primary ray is regenerated on the owner from the global pixel index, the
 * camera, the AOV call's seed, first_sample and RT3_FLAG_NO_JITTER, which the fingerprints prove every part shared, so
 * the owner reprojects rows it did not render. The history is the owner's rt3_denoise_temporal history, with the same
 * rules: dropped on reset, when there is none, or when the size or the owner's scene upload differ, and kept only when
 * a call succeeds. Every part must therefore upload a new scene when the owner does. For each frame of a sequence the
 * result (host_frame, host_rgb, host_history_length; any may be NULL) is bit-equal to rt3_denoise_temporal over
 * one-context renders of the same frames, so a sequence may mix both calls on the owner's context and still gives the
 * bits of an all-one-context sequence; a call with no usable history is bit-equal to rt3_denoise_staged. Blocking. A
 * refused call (RT3_ERR_INVALID) changes nothing, the stage and the history included; a CUDA error drops the history.
 * The accumulators, the AOV buffers and the RT3_FLAG_ACCUMULATE state are only read; rt3_get_stats then describes this
 * call (device_ms, kernel_launches = 2 + iterations, rays = 0). */
int rt3_denoise_staged_temporal(rt3_ctx* ctx, const rt3_denoise_temporal_params* params, uint64_t frame_tag, const uint32_t* device_stage,
                                uint32_t* host_frame, float* host_rgb, float* host_history_length);

/* Device-resident variant for multi-GPU plumbing: renders this partition's
 * rows into `device_frame` (a device pointer to width*height uint32, full-frame
 * indexing) asynchronously on `cuda_stream` (a cudaStream_t; NULL = the
 * context's own stream). No host copies, and the call does not wait for the render. It is not entirely free
 * of synchronisation: the first RT3_FLAG_BVH render after an upload builds the hierarchy and waits for it, and
 * when several contexts on one device take turns with scenes small enough for the constant bank
 * (<= 768 primitives), a change of turn waits for the device to drain before the records are swapped.
 * Contexts may be driven from different host threads (one thread per context at a time). */
int rt3_render_device(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, uint32_t* device_frame,
                      void* cuda_stream);

/* Number of rows `part_index` owns under (height, tile_rows, part_count), and
 * packing/unpacking between full-frame row order and a partition's compact
 * slab (its owned rows, top to bottom) for the frame-end gather. Both run on
 * the device, asynchronously on `cuda_stream`. */
uint32_t rt3_partition_rows(uint32_t height, uint32_t tile_rows, uint32_t part_index, uint32_t part_count);
int rt3_pack_partition(rt3_ctx* ctx, const uint32_t* device_frame, uint32_t* device_slab, uint32_t width, uint32_t height,
                       uint32_t tile_rows, uint32_t part_index, uint32_t part_count, void* cuda_stream);
int rt3_unpack_partition(rt3_ctx* ctx, const uint32_t* device_slab, uint32_t* device_frame, uint32_t width, uint32_t height,
                         uint32_t tile_rows, uint32_t part_index, uint32_t part_count, void* cuda_stream);

/* Shared frame for the multi-GPU split (SURVEY.md section 8e; the reference's hook is the unused BlockInfo
 * uniform, src/lib/shaders/raytracer/raytracer_v4.glsl:70-79). One process allocates the full frame on its
 * GPU (rt3_frame_alloc) and exports it (rt3_frame_export, a CUDA IPC handle of RT3_IPC_HANDLE_BYTES bytes
 * that travels over any channel); every other process maps it (rt3_frame_import, peer access over NVLink is
 * enabled on first use) and passes the mapped pointer to rt3_render_device as `device_frame`. Frames use
 * full-frame indexing, so each partition's kernels store its rows where they belong in the owner's memory:
 * the frame-end gather is the render kernels' own stores, and all that is left is a barrier. A process that
 * imported a frame releases it (rt3_frame_release) before the owner frees it (rt3_frame_free). */
#define RT3_IPC_HANDLE_BYTES 64
int rt3_frame_alloc(rt3_ctx* ctx, uint64_t n_pixels, uint32_t** device_frame);
int rt3_frame_free(rt3_ctx* ctx, uint32_t* device_frame);
int rt3_frame_export(rt3_ctx* ctx, const uint32_t* device_frame, unsigned char* handle_out);
int rt3_frame_import(rt3_ctx* ctx, const unsigned char* handle, uint32_t** peer_frame);
int rt3_frame_release(rt3_ctx* ctx, uint32_t* peer_frame);
/* Same sharing inside one process (several contexts, one per GPU): rt3_frame_attach lets `ctx`'s device store into
 * frames that live on `owner`'s device (peer access; nothing to do when the two are one device), after which a
 * pointer from rt3_frame_alloc(owner) is a valid `device_frame` for rt3_render_device(ctx). rt3_frame_read copies
 * n_pixels packed pixels of a device frame into host memory and returns when they are there. */
int rt3_frame_attach(rt3_ctx* ctx, rt3_ctx* owner);
int rt3_frame_read(rt3_ctx* ctx, const uint32_t* device_frame, uint32_t* host_frame, uint64_t n_pixels);

/* Scene construction on the device (the step before the path): tessellates `n` UV spheres with the arithmetic of
 * the reference's CPU pre-render (src/lib/entities/Sphere.cpp:69-79,120-351; GPU twins
 * shaders/pre_render_sphere_v2_{vertices,faces}.glsl) and returns them flattened like
 * SequentialRenderer.cpp:174-195: sphere k's vertices follow sphere k-1's, face indices are absolute,
 * shifted by `first_vertex` (where the caller appends the batch in its own vertex array). The host arrays must
 * hold the sums of rt3_uv_sphere_faces / rt3_uv_sphere_vertices; host_face_entity may be NULL. */
uint32_t rt3_uv_sphere_faces(uint32_t n_meridians, uint32_t n_parallels);
uint32_t rt3_uv_sphere_vertices(uint32_t n_meridians, uint32_t n_parallels);
int rt3_tessellate_spheres(rt3_ctx* ctx, const rt3_uv_sphere* spheres, uint32_t n, uint32_t first_vertex, rt3_face* host_faces,
                           rt3_vertex* host_vertices, uint32_t* host_face_entity);
/* The same without the trip to the host: the batch is written into DEVICE arrays the caller owns, sphere k's vertices
 * from device_vertices[first_vertex] on and its faces from device_faces[first_face] on, face indices absolute (they index
 * device_vertices). device_face_entity may be NULL. Asynchronous on the context's stream, which rt3_scene_upload_device
 * and rt3_buffer_* also use, so the calls order themselves. */
int rt3_tessellate_spheres_device(rt3_ctx* ctx, const rt3_uv_sphere* spheres, uint32_t n, uint32_t first_vertex, uint32_t first_face,
                                  rt3_face* device_faces, rt3_vertex* device_vertices, uint32_t* device_face_entity);

/* Output side (the step after the path, reference camera/Frame.cpp:88-96,131-142): unpacks a device frame of
 * width*height packed pixels into interleaved 8-bit RGB (channels = 3) or RGBA (channels = 4, alpha 255) bytes,
 * the layout PPM / PNG writers take, on the device and asynchronously on `cuda_stream`. Both pointers are
 * device pointers, 16-byte aligned. */
int rt3_frame_bytes(rt3_ctx* ctx, const uint32_t* device_frame, unsigned char* device_out, uint32_t width, uint32_t height, uint32_t channels,
                    void* cuda_stream);

/* Float AOV of the last path-traced render on this context: the mean linear radiance behind the frame (the value the
 * resolve takes the square root of and packs, reference packing SequentialRenderer.cpp:297), 3 floats (r, g, b) per pixel,
 * width * height pixels in frame order (the size of that render, checked); rows of other partitions are 0. Blocking. */
int rt3_read_radiance(rt3_ctx* ctx, float* host_rgb, uint32_t width, uint32_t height);

int rt3_get_stats(rt3_ctx* ctx, rt3_stats* out);

/* Achieved FP32 FMA throughput of a dependent-chain-free FFMA micro-kernel on
 * this context's device, in TFLOP/s (2 FLOP per FMA): the measured
 * denominator for the roofline fraction. */
int rt3_measure_fma_peak(rt3_ctx* ctx, double* tflops_out);

#ifdef __cplusplus
}
#endif

#endif /* RT3CUDA_H */
