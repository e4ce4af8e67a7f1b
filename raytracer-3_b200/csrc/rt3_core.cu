/* rt3_core.cu — host side of librt3cuda.so: the C ABI of include/rt3cuda.h.
 *
 * Owns one CUDA context per rt3_ctx: the flattened scene in HBM (SoA), the
 * frame / AOV / accumulator buffers, a stream and the timing events. Scene
 * upload mirrors what the reference's GPU backend does in prerender
 * (reference src/lib/renderer/VulkanRenderer.cpp:266-399: flatten once, keep
 * on the device, reuse across render() calls); render mirrors
 * VulkanRenderer.cpp:402-557 without its per-call pipeline rebuild.
 *
 * Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false
 * (see __graft_entry__.build()). There is no CPU path in this library.
 */
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <limits>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "rt3_kernels.cuh"
#include "rt3_denoise.cuh"
#include "rt3_scene.cuh"
#include "rt3_upload.cuh"

namespace {

thread_local std::string g_error;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define RT3_CUDA(call)                                                                                           \
    do {                                                                                                         \
        cudaError_t e__ = (call);                                                                                \
        if (e__ != cudaSuccess) {                                                                                \
            (void) cudaGetLastError(); /* reported here: must not resurface at a later launch check */         \
            return fail(RT3_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__));                        \
        }                                                                                                        \
    } while (0)

/* Device allocation owned by its holder: context members live as long as the context, scratch
 * buffers of one call are freed on every way out of it. */
template <class T> struct DeviceBuffer {
    T* ptr = nullptr;
    size_t count = 0;
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    ~DeviceBuffer() { release(); }
    int reserve(size_t n) {
        if (n <= count) { return RT3_OK; }
        if (ptr) { cudaFree(ptr); ptr = nullptr; count = 0; }
        RT3_CUDA(cudaMalloc(&ptr, n * sizeof(T)));
        count = n;
        return RT3_OK;
    }
    void release() { if (ptr) { cudaFree(ptr); } ptr = nullptr; count = 0; }
};

/* A pair of timing events that does not outlive the call that made it. */
struct EventPair {
    cudaEvent_t begin = nullptr, end = nullptr;
    EventPair() = default;
    EventPair(const EventPair&) = delete;
    EventPair& operator=(const EventPair&) = delete;
    ~EventPair() { if (begin) { cudaEventDestroy(begin); } if (end) { cudaEventDestroy(end); } }
    int create() {
        RT3_CUDA(cudaEventCreate(&begin));
        RT3_CUDA(cudaEventCreate(&end));
        return RT3_OK;
    }
};

}  // namespace

struct rt3_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_copy = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;
    cudaStream_t last_stream = nullptr; /* stream of the most recent render */
    bool stats_pending = false;         /* timings / counters not yet read back */
    bool stats_beam_accel = false;      /* ... or, through the hierarchy, against the candidates a beam's walk of the trees collected (counters[5], [6]) */
    bool stats_beam = false;            /* the most recent render traced its primary rays against candidate lists (counters[2], [3]) */
    bool copy_timed = false;

    bool has_scene = false;
    rt3_scene_view view{};
    uint64_t scene_id = 0; /* identifies the uploaded scene as owner of the constant-bank records */
    DeviceBuffer<float4> pair_xy, filt3, face_rec, spheres, prim_color, materials;
    DeviceBuffer<float2> pair_w;
    DeviceBuffer<uint32_t> prim_material, prim_entity;

    /* hierarchy (RT3_FLAG_BVH): primitive boxes are uploaded with the scene, the tree is built on first use */
    DeviceBuffer<float4> prim_lo, prim_hi, bvh_nodes;
    float centroid_min[3] = { 0, 0, 0 }, centroid_max[3] = { 0, 0, 0 };
    bool bvh_ready = false;
    rt3_bvh_view bvh{};
    double bvh_build_ms = 0.0;

    DeviceBuffer<uint32_t> frame, aov_prim, aov_entity;
    DeviceBuffer<float> aov_t;
    DeviceBuffer<unsigned long long> aov_sums; /* rt3_render_path_aovs: RT3_AOV_SUMS per pixel, apart from the path tracer's accumulators */
    DeviceBuffer<float> aov_albedo, aov_normal;
    DeviceBuffer<unsigned long long> accum, counters;
    rt3_kparams accum_kp{};                      /* the path-traced render the accumulators currently hold */
    bool accum_valid = false;
    uint32_t accum_first = 0;                    /* the first sample it holds (rt3_denoise_stage's fingerprint) */
    rt3_camera accum_cam{};                      /* its camera (rt3_denoise) ... */
    bool accum_cam_mixed = false;                /* ... unless an accumulating pass used another one */

    /* the last rt3_render_path_aovs, whose albedo, normal and depth (aov_t) guide rt3_denoise */
    bool path_aovs_valid = false;
    rt3_kparams path_aovs_kp{};
    rt3_camera path_aovs_cam{};
    uint64_t path_aovs_scene_id = 0;

    /* rt3_denoise: ping-pong filter state, guides and outputs, sized on first use */
    DeviceBuffer<rt3_dn_px> dn_col[2];
    DeviceBuffer<rt3_dn_guide> dn_guide;
    DeviceBuffer<float> dn_rgb;
    DeviceBuffer<uint32_t> dn_frame;

    /* rt3_denoise_temporal: two histories, the valid one read and the other written; they swap when a call succeeds. The
     * camera, size and scene upload are those of the frame that produced the valid one. */
    DeviceBuffer<rt3_dn_hist> dn_hist_col[2];
    DeviceBuffer<rt3_dn_moments> dn_hist_mom[2];
    DeviceBuffer<rt3_dn_guide> dn_hist_guide[2];
    DeviceBuffer<float> dn_hist_length;
    uint32_t dn_hist_cur = 0;
    bool dn_hist_valid = false;
    rt3_camera dn_hist_cam{};
    uint32_t dn_hist_width = 0, dn_hist_height = 0;
    uint64_t dn_hist_scene_id = 0;

    rt3_stats stats{};
    double upload_ms = 0.0, upload_h2d_ms = 0.0, upload_device_ms = 0.0; /* most recent scene upload */
};

namespace {

uint32_t owned_rows(uint32_t height, uint32_t tile_rows, uint32_t part_index, uint32_t part_count) {
    if (tile_rows == 0) { tile_rows = 1; }
    if (part_count <= 1) { return height; }
    uint32_t n_tiles = (height + tile_rows - 1) / tile_rows, rows = 0;
    for (uint32_t t = part_index; t < n_tiles; t += part_count) {
        uint32_t first = t * tile_rows;
        rows += (height - first < tile_rows) ? height - first : tile_rows;
    }
    return rows;
}

int make_kparams(const rt3_params* p, rt3_kparams* k) {
    if (!p) { return fail(RT3_ERR_INVALID, "params is NULL"); }
    if (p->width < 2 || p->height < 2) { return fail(RT3_ERR_INVALID, "frame must be at least 2x2 (got %ux%u)", p->width, p->height); }
    if ((unsigned long long) p->width * p->height > 0xFFFFFFFFull) { return fail(RT3_ERR_INVALID, "frame too large"); }
    if (p->mode != RT3_MODE_REFERENCE && p->mode != RT3_MODE_PATHTRACE) { return fail(RT3_ERR_INVALID, "unknown mode %u", p->mode); }
    if (p->mode == RT3_MODE_PATHTRACE && (p->spp < 1 || p->spp > 65535 || p->max_depth < 1)) {
        return fail(RT3_ERR_INVALID, "pathtrace needs 1 <= spp <= 65535 and max_depth >= 1 (got spp %u, depth %u)", p->spp, p->max_depth);
    }
    uint32_t parts = p->part_count ? p->part_count : 1;
    if (p->part_index >= parts) { return fail(RT3_ERR_INVALID, "part_index %u >= part_count %u", p->part_index, parts); }
    k->width = p->width; k->height = p->height;
    k->spp = p->mode == RT3_MODE_PATHTRACE ? p->spp : 1;
    k->first_sample = p->mode == RT3_MODE_PATHTRACE ? p->first_sample : 0;
    if ((unsigned long long) k->first_sample + k->spp > 0x7FFFFFFFull) { return fail(RT3_ERR_INVALID, "first_sample + spp must stay below 2^31"); }
    k->resolve_spp = (p->flags & RT3_FLAG_ACCUMULATE) ? k->first_sample + k->spp : k->spp;
    k->max_depth = p->max_depth; k->seed = p->seed; k->flags = p->flags;
    k->tile_rows = p->tile_rows ? p->tile_rows : 1;
    k->part_index = p->part_index; k->part_count = parts;
    k->owned_rows = owned_rows(p->height, k->tile_rows, p->part_index, parts);
    k->n_pixels = (unsigned long long) k->owned_rows * p->width;
    k->n_items = k->n_pixels * k->spp;
    k->resident = 0;
    return RT3_OK;
}

/* Which scene owns the constant-bank records of each device (rt3_device.cuh c_pair_xy / c_pair_w).
 * One mutex per device, held from the claim until the kernel that reads the bank has been enqueued: a
 * later claim by another context then waits for that kernel (cudaDeviceSynchronize under the same
 * mutex) before it overwrites the records. */
constexpr int RT3_MAX_DEVICES = 64;
std::mutex g_const_mutex[RT3_MAX_DEVICES];
uint64_t g_const_owner[RT3_MAX_DEVICES] = { 0 };
std::atomic<uint64_t> g_next_scene_id{ 1 };

template <class K> int configure(K kernel, size_t smem, int* blocks_per_sm) {
    RT3_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    if (blocks_per_sm) { RT3_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, kernel, RT3_CTA_THREADS, smem)); }
    return RT3_OK;
}

template <bool RESIDENT, bool SPHERES_ONLY, bool ACCEL>
int launch_reference(rt3_ctx* ctx, const rt3_camera& cam, const rt3_kparams& kp, size_t smem, uint32_t* frame, uint32_t* prim,
                     uint32_t* ent, float* t, cudaStream_t stream) {
    int rc = configure(reference_kernel<RESIDENT, SPHERES_ONLY, ACCEL>, smem, nullptr);
    if (rc != RT3_OK) { return rc; }
    unsigned long long per_cta = (unsigned long long) RT3_CTA_THREADS * RT3_REF_RAYS;
    unsigned grid = (unsigned) ((kp.n_pixels + per_cta - 1) / per_cta);
    reference_kernel<RESIDENT, SPHERES_ONLY, ACCEL><<<grid, RT3_CTA_THREADS, smem, stream>>>(ctx->view, ctx->bvh, cam, kp, frame, prim, ent, t, ctx->counters.ptr);
    RT3_CUDA(cudaGetLastError());
    return RT3_OK;
}

template <bool RESIDENT, bool SPHERES_ONLY, bool ACCEL, int BIN = 0, bool BEAM = false>
int launch_pathtrace(rt3_ctx* ctx, const rt3_camera& cam, const rt3_kparams& kp, size_t smem, cudaStream_t stream) {
    int per_sm = 0;
    int rc = configure(pathtrace_kernel<RESIDENT, SPHERES_ONLY, ACCEL, BIN, BEAM>, smem, &per_sm);
    if (rc != RT3_OK) { return rc; }
    if (ACCEL) {
        /* The traversal reads its node records through L1: ask for the smallest shared-memory carve-out that still
         * holds the resident CTAs (1 KB of system use each) -- the default rounds up one configuration further. */
        int sm_bytes = 0;
        RT3_CUDA(cudaDeviceGetAttribute(&sm_bytes, cudaDevAttrMaxSharedMemoryPerMultiprocessor, ctx->device));
        const size_t need = (size_t) per_sm * (smem + 1024);
        int percent = sm_bytes > 0 ? (int) ((need * 100 + (size_t) sm_bytes - 1) / (size_t) sm_bytes) : 100;
        if (percent > 100) { percent = 100; }
        RT3_CUDA(cudaFuncSetAttribute(pathtrace_kernel<RESIDENT, SPHERES_ONLY, ACCEL, BIN, BEAM>, cudaFuncAttributePreferredSharedMemoryCarveout, percent));
    }
    if (per_sm < 1) { return fail(RT3_ERR_CUDA, "pathtrace kernel does not fit on an SM (smem %zu)", smem); }
    if (const char* cap = getenv("RT3_MAX_CTAS_PER_SM")) { /* tuning knob: fewer persistent CTAs per SM than fit */
        const int c = atoi(cap);
        if (c >= 1 && c < per_sm) { per_sm = c; }
    }
    /* persistent grid: every SM full, no more CTAs than there are CTAs' worth of paths */
    unsigned long long per_cta = (unsigned long long) RT3_CTA_THREADS * RT3_RAYS;
    unsigned long long want = (kp.n_items + per_cta - 1) / per_cta;
    unsigned grid = (unsigned) ctx->sm_count * (unsigned) per_sm;
    if (want < grid) { grid = want ? (unsigned) want : 1u; }
    pathtrace_kernel<RESIDENT, SPHERES_ONLY, ACCEL, BIN, BEAM><<<grid, RT3_CTA_THREADS, smem, stream>>>(ctx->view, ctx->bvh, cam, kp, ctx->accum.ptr, ctx->counters.ptr);
    RT3_CUDA(cudaGetLastError());
    return RT3_OK;
}

template <bool RESIDENT, bool SPHERES_ONLY, bool ACCEL>
int launch_path_aovs(rt3_ctx* ctx, const rt3_camera& cam, const rt3_kparams& kp, size_t smem, uint32_t* prim, uint32_t* ent, float* t,
                     cudaStream_t stream) {
    int rc = configure(path_aov_kernel<RESIDENT, SPHERES_ONLY, ACCEL>, smem, nullptr);
    if (rc != RT3_OK) { return rc; }
    const unsigned long long per_cta = (unsigned long long) RT3_CTA_THREADS * RT3_REF_RAYS;
    const unsigned long long grid = (kp.n_items + per_cta - 1) / per_cta;
    if (grid > 0x7FFFFFFFull) { return fail(RT3_ERR_INVALID, "too many AOV samples in one call (%llu)", kp.n_items); }
    path_aov_kernel<RESIDENT, SPHERES_ONLY, ACCEL><<<(unsigned) grid, RT3_CTA_THREADS, smem, stream>>>(ctx->view, ctx->bvh, cam, kp, ctx->aov_sums.ptr, prim, ent, t,
                                                                                                     ctx->counters.ptr);
    RT3_CUDA(cudaGetLastError());
    return RT3_OK;
}

/* Builds the hierarchy over the uploaded primitive boxes (first RT3_FLAG_BVH render after an upload):
 * Morton codes of the box centres, radix sort (CUB), Karras' radix tree, bottom-up refit. All on the
 * device; the scratch arrays are released when the node array is complete.
 * Faces and spheres get a tree each (one node array, the sphere tree's nodes behind the face tree's):
 * the sphere discriminant needs boxes widened by sqrt(2^-18)|o| per ray, and that much around the
 * small triangles of a tessellated mesh makes every ray that starts on the mesh walk its whole
 * neighbourhood. The face tree's per-ray widening only covers the rounding of the slab test itself. */
int build_bvh(rt3_ctx* ctx, cudaStream_t stream) {
    if (ctx->bvh_ready) { return RT3_OK; }
    const uint32_t count[2] = { ctx->view.n_faces, ctx->view.n_spheres }, first[2] = { 0u, ctx->view.n_faces };
    /* per-ray widening (times |o|): a few 2^-24 for the triangle test's hit point and the slab test's own o / d
     * product (2^-19 in all), sqrt(2^-18) for the sphere discriminant */
    const float margin[2] = { 1.9073486328125e-06f, sqrtf(RT3_FILTER_SLACK) * 1.0001f };
    ctx->bvh.n_prims = ctx->view.n_prims;
    ctx->bvh.nodes = nullptr;
    ctx->bvh_build_ms = 0.0;
    uint32_t node_offset[2] = { 0u, count[0] > 1 ? count[0] - 1 : 0u };
    const size_t n_nodes = (size_t) node_offset[1] + (count[1] > 1 ? count[1] - 1 : 0u);
    for (int w = 0; w < 2; w++) {
        ctx->bvh.tree[w].n_prims = count[w];
        ctx->bvh.tree[w].root = count[w] == 1 ? ~(int32_t) first[w] : (int32_t) node_offset[w];
        ctx->bvh.tree[w].ray_margin = margin[w];
    }
    const uint32_t nmax = count[0] > count[1] ? count[0] : count[1];
    if (nmax < 2) { ctx->bvh_ready = true; return RT3_OK; }
    DeviceBuffer<unsigned long long> keys_in, keys_out;
    DeviceBuffer<uint32_t> vals_in, vals_out, arrived;
    DeviceBuffer<int> child, node_parent, leaf_parent;
    DeviceBuffer<float4> box_lo, box_hi;
    DeviceBuffer<unsigned char> temp;
    int rc;
    if ((rc = keys_in.reserve(nmax)) != RT3_OK || (rc = keys_out.reserve(nmax)) != RT3_OK || (rc = vals_in.reserve(nmax)) != RT3_OK ||
        (rc = vals_out.reserve(nmax)) != RT3_OK || (rc = arrived.reserve(nmax)) != RT3_OK || (rc = child.reserve(2 * (size_t) nmax)) != RT3_OK ||
        (rc = node_parent.reserve(nmax)) != RT3_OK || (rc = leaf_parent.reserve(nmax)) != RT3_OK || (rc = box_lo.reserve(nmax)) != RT3_OK ||
        (rc = box_hi.reserve(nmax)) != RT3_OK || (rc = ctx->bvh_nodes.reserve(4 * (n_nodes ? n_nodes : 1))) != RT3_OK) {
        return rc;
    }
    size_t temp_bytes = 0;
    RT3_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys_in.ptr, keys_out.ptr, vals_in.ptr, vals_out.ptr, (int) nmax, 0, 63, stream));
    if ((rc = temp.reserve(temp_bytes ? temp_bytes : 1)) != RT3_OK) { return rc; }
    float3 cmin = make_float3(ctx->centroid_min[0], ctx->centroid_min[1], ctx->centroid_min[2]), cscale;
    {
        const float ex[3] = { ctx->centroid_max[0] - ctx->centroid_min[0], ctx->centroid_max[1] - ctx->centroid_min[1],
                              ctx->centroid_max[2] - ctx->centroid_min[2] };
        cscale = make_float3(ex[0] > 0 ? 1.0f / ex[0] : 0.0f, ex[1] > 0 ? 1.0f / ex[1] : 0.0f, ex[2] > 0 ? 1.0f / ex[2] : 0.0f);
    }
    EventPair ev;
    if ((rc = ev.create()) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ev.begin, stream));
    for (int w = 0; w < 2; w++) {
        const uint32_t n = count[w];
        if (n < 2) { continue; }
        const unsigned grid = (n + 255u) / 256u;
        bvh_morton_kernel<<<grid, 256, 0, stream>>>(n, first[w], ctx->prim_lo.ptr, ctx->prim_hi.ptr, cmin, cscale, keys_in.ptr, vals_in.ptr);
        RT3_CUDA(cudaGetLastError());
        size_t tb = temp_bytes;
        RT3_CUDA(cub::DeviceRadixSort::SortPairs(temp.ptr, tb, keys_in.ptr, keys_out.ptr, vals_in.ptr, vals_out.ptr, (int) n, 0, 63, stream));
        RT3_CUDA(cudaMemsetAsync(arrived.ptr, 0, (size_t) n * sizeof(uint32_t), stream));
        bvh_tree_kernel<<<grid, 256, 0, stream>>>((int) n, keys_out.ptr, child.ptr, node_parent.ptr, leaf_parent.ptr);
        RT3_CUDA(cudaGetLastError());
        bvh_refit_kernel<<<grid, 256, 0, stream>>>((int) n, vals_out.ptr, ctx->prim_lo.ptr, ctx->prim_hi.ptr, child.ptr, node_parent.ptr, leaf_parent.ptr,
                                                  box_lo.ptr, box_hi.ptr, arrived.ptr, ctx->bvh_nodes.ptr, (int) node_offset[w]);
        RT3_CUDA(cudaGetLastError());
    }
    RT3_CUDA(cudaEventRecord(ev.end, stream));
    RT3_CUDA(cudaStreamSynchronize(stream)); /* the scratch arrays go out of scope */
    float ms = 0.f;
    RT3_CUDA(cudaEventElapsedTime(&ms, ev.begin, ev.end));
    ctx->bvh_build_ms = ms;
    ctx->bvh.nodes = ctx->bvh_nodes.ptr;
    ctx->bvh_ready = true;
    return RT3_OK;
}

/* Makes this context's scene the owner of the device's constant-bank records. The bank is one per
 * device and module, so a change of owner waits for everything in flight on the device, copies the
 * records (device to device) and waits for the copy; renders of one scene never pay this.
 * `lock` is taken here and stays with the caller until its kernel launch has been enqueued. */
int claim_constant_bank(rt3_ctx* ctx, cudaStream_t stream, std::unique_lock<std::mutex>& lock) {
    if (ctx->device < 0 || ctx->device >= RT3_MAX_DEVICES) { return fail(RT3_ERR_INVALID, "device %d out of range", ctx->device); }
    lock = std::unique_lock<std::mutex>(g_const_mutex[ctx->device]);
    if (g_const_owner[ctx->device] == ctx->scene_id) { return RT3_OK; }
    RT3_CUDA(cudaDeviceSynchronize());
    const size_t pairs = ctx->view.n_prims_padded / 2;
    if (pairs) {
        RT3_CUDA(cudaMemcpyToSymbolAsync(c_pair_xy, ctx->pair_xy.ptr, pairs * sizeof(float4), 0, cudaMemcpyDeviceToDevice, stream));
        RT3_CUDA(cudaMemcpyToSymbolAsync(c_pair_w, ctx->pair_w.ptr, pairs * sizeof(float2), 0, cudaMemcpyDeviceToDevice, stream));
    }
    RT3_CUDA(cudaStreamSynchronize(stream));
    g_const_owner[ctx->device] = ctx->scene_id;
    return RT3_OK;
}

/* How a kernel traces the uploaded scene: through the hierarchy, or by sweeping the primitive records from the
 * constant bank (resident) or streamed from HBM; and the dynamic shared memory that takes. */
struct trace_plan { bool accel, resident, spheres_only; size_t smem; };

/* The plan for a trace with `flags` (RT3_FLAG_BVH); builds the hierarchy on its first use after an upload. `path_slots`:
 * the kernel keeps path state in shared memory (the path tracer). */
int plan_trace(rt3_ctx* ctx, uint32_t flags, bool path_slots, cudaStream_t stream, trace_plan* plan) {
    plan->accel = (flags & RT3_FLAG_BVH) != 0;
    plan->spheres_only = ctx->view.n_faces == 0;
    if (plan->accel) {
        plan->resident = false; /* no constant-bank records needed */
        plan->smem = rt3_accel_smem_bytes(path_slots);
        return build_bvh(ctx, stream);
    }
    plan->resident = ctx->view.n_prims_padded <= RT3_CONST_PRIMS;
    plan->smem = rt3_smem_bytes(plan->resident, path_slots);
    return RT3_OK;
}

/* Calls f(RESIDENT, SPHERES_ONLY, ACCEL), each a std::integral_constant<bool>, for the plan's instantiation of a
 * trace kernel. Each kernel exists in five variants: the hierarchy's <true, false, true>, and the sweep's over the
 * constant bank or streamed tiles, with or without faces. */
template <class F> int with_scene_variant(const trace_plan& plan, F&& f) {
    using Y = std::true_type; using N = std::false_type;
    if (plan.accel) { return f(Y{}, N{}, Y{}); }
    if (plan.resident) { return plan.spheres_only ? f(Y{}, Y{}, N{}) : f(Y{}, N{}, N{}); }
    return plan.spheres_only ? f(N{}, Y{}, N{}) : f(N{}, N{}, N{});
}

/* Starts a pass on `stream`: from here on the statistics collect_stats reads back are this pass's. With `bank_lock`,
 * the scene is made the constant bank's owner first, and the lock stays with the caller until its kernel has been
 * enqueued. The pass's timing and counters start after the claim. */
int begin_pass(rt3_ctx* ctx, bool accel, uint32_t rows, cudaStream_t stream, std::unique_lock<std::mutex>* bank_lock) {
    ctx->stats.accel = accel ? 1u : 0u;
    ctx->stats_beam = false; ctx->stats_beam_accel = false;
    ctx->stats.kernel_launches = 0;
    ctx->stats.rows_rendered = rows;
    ctx->last_stream = stream;
    ctx->stats_pending = true;
    ctx->copy_timed = false;
    int rc;
    if (bank_lock && (rc = claim_constant_bank(ctx, stream, *bank_lock)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_begin, stream));
    RT3_CUDA(cudaMemsetAsync(ctx->counters.ptr, 0, 8 * sizeof(unsigned long long), stream));
    return RT3_OK;
}

/* Ends a blocking pass: times the device-to-host copies enqueued after ev_end and waits for them. */
int end_pass(rt3_ctx* ctx, cudaStream_t stream) {
    RT3_CUDA(cudaEventRecord(ctx->ev_copy, stream));
    ctx->copy_timed = true;
    RT3_CUDA(cudaStreamSynchronize(stream));
    return RT3_OK;
}

/* Enqueues one render of this partition into device_frame (full-frame indexing). */
int enqueue_render(rt3_ctx* ctx, const rt3_camera* cam, const rt3_params* params, const rt3_kparams& kp_in, uint32_t* device_frame,
                   uint32_t* prim, uint32_t* ent, float* t, cudaStream_t stream) {
    rt3_kparams kp = kp_in;
    if (params->mode == RT3_MODE_PATHTRACE && (params->flags & RT3_FLAG_ACCUMULATE)) {
        /* checked before anything of the previous render (its statistics, its events) is touched */
        const rt3_kparams& prev = ctx->accum_kp;
        if (!ctx->accum_valid || prev.width != kp.width || prev.height != kp.height) {
            return fail(RT3_ERR_INVALID, "RT3_FLAG_ACCUMULATE needs a previous path-traced render of the same %ux%u frame and scene on this context", kp.width, kp.height);
        }
        if (prev.tile_rows != kp.tile_rows || prev.part_index != kp.part_index || prev.part_count != kp.part_count) {
            return fail(RT3_ERR_INVALID, "RT3_FLAG_ACCUMULATE: partition (tile_rows %u, part %u of %u) differs from the accumulated render's (%u, %u of %u)",
                        kp.tile_rows, kp.part_index, kp.part_count, prev.tile_rows, prev.part_index, prev.part_count);
        }
        if (prev.seed != kp.seed || prev.max_depth != kp.max_depth || ((prev.flags ^ kp.flags) & ~(RT3_FLAG_ACCUMULATE | RT3_FLAG_BVH | RT3_FLAG_NO_GAMMA))) {
            return fail(RT3_ERR_INVALID, "RT3_FLAG_ACCUMULATE: seed, max_depth and sampling flags must be those of the accumulated render");
        }
        if (kp.first_sample != prev.first_sample + prev.spp) {
            return fail(RT3_ERR_INVALID, "RT3_FLAG_ACCUMULATE: first_sample must continue the accumulated range (expected %u, got %u)", prev.first_sample + prev.spp, kp.first_sample);
        }
    }
    trace_plan plan;
    int rc = plan_trace(ctx, params->flags, params->mode == RT3_MODE_PATHTRACE, stream, &plan);
    if (rc != RT3_OK) { return rc; }
    kp.resident = plan.resident ? 1u : 0u;
    std::unique_lock<std::mutex> bank_lock; /* released when this function returns, i.e. after the launch below */
    if ((rc = begin_pass(ctx, plan.accel, kp.owned_rows, stream, plan.resident && kp.n_pixels != 0 ? &bank_lock : nullptr)) != RT3_OK) { return rc; }
    if (kp.n_pixels == 0) {
        RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
        RT3_CUDA(cudaEventRecord(ctx->ev_k1, stream));
        RT3_CUDA(cudaEventRecord(ctx->ev_end, stream));
        return RT3_OK;
    }
    if (params->mode == RT3_MODE_REFERENCE) {
        RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
        rc = with_scene_variant(plan, [&](auto r, auto so, auto a) {
            return launch_reference<decltype(r)::value, decltype(so)::value, decltype(a)::value>(ctx, *cam, kp, plan.smem, device_frame, prim, ent, t, stream);
        });
        if (rc != RT3_OK) { return rc; }
        RT3_CUDA(cudaEventRecord(ctx->ev_k1, stream));
        RT3_CUDA(cudaEventRecord(ctx->ev_end, stream));
        ctx->stats.kernel_launches = 1;
        return rc;
    }
    size_t n_acc = (size_t) kp.width * kp.height * 3;
    const bool accumulate = (params->flags & RT3_FLAG_ACCUMULATE) != 0;
    if (!accumulate) {
        ctx->accum_valid = false;
        rc = ctx->accum.reserve(n_acc);
        if (rc != RT3_OK) { return rc; }
        unsigned clear_grid = (unsigned) ((kp.n_pixels * 3ull + 255ull) / 256ull);
        clear_accum_kernel<<<clear_grid, 256, 0, stream>>>(kp, ctx->accum.ptr);
        RT3_CUDA(cudaGetLastError());
    }
    RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
    /* scenes with a real face tree sort their rays by whether they enter it (rt3_kernels.cuh traverse_slots_binned) */
    int bin = 0; /* 0 none, 1 CTA-wide, 2 / 3 per warp with two / three classes */
    if (plan.accel && ctx->bvh.tree[0].n_prims >= RT3_BIN_MIN_FACES && ctx->bvh.tree[0].root >= 0) {
        /* Measured on C3 (profiles/r02e_variants.jsonl; none / CTA-wide / per warp): 256 spp 365 / 399 / 343 ms, 16 spp 28.7 / 27.8 / 27.3,
         * 4 spp 10.4 / 8.9 / 9.6. The CTA-wide sort pays when a warp's rays come from many pixels (few samples per pixel and call:
         * interactive / progressive passes) and costs 9 % at 256 spp, where a warp's rays share a pixel and the barriers only cost;
         * the per-warp sort needs no barrier and gains 5-8 % everywhere; with a third class in front (rays that START inside the root box:
         * bounces off the mesh) another 2.5-4 % (profiles/r02x_variants.jsonl: 256 spp 333.8 -> 325.3 ms, 16 spp 25.9 -> 24.8). */
        bin = kp.spp <= RT3_BIN_MAX_SPP ? 1 : 3;
        if (const char* e = getenv("RT3_BINNING")) { bin = atoi(e); } /* for A/B measurements */
    }
    /* resident sphere scenes: primary rays are traced against a per-chunk candidate list instead of the sweep (rt3_kernels.cuh, "BEAM");
     * RT3_BEAM=0 switches it off for A/B measurements */
    bool beam = !plan.accel && plan.resident && plan.spheres_only;
    if (const char* e = getenv("RT3_BEAM")) { beam = beam && atoi(e) != 0; }
    /* the same through the hierarchy (the beam walks the trees once per chunk of path items): the unsorted hierarchy kernel, i.e. sphere scenes and
     * small meshes. Measured (call AG, profiles/r02ag_variants.jsonl): C5 45.7 -> 27.5 ms (17.0 after calls AH, AI), C2 through the hierarchy 129.4 -> 117.4 ms; under the sorted
     * traversal of large meshes it gains nothing (C3 325.1 -> 327.8 ms: the primary rays of such a scene are its cheap rays, and the warp-wide
     * regeneration the beams need is the slower one there), so that kernel takes it only on request: RT3_BEAM_BVH=1 (0: never) */
    bool beam_accel = plan.accel && bin == 0;
    if (const char* e = getenv("RT3_BEAM_BVH")) { beam_accel = plan.accel && (bin == 0 || bin == 3) && atoi(e) != 0; }
    if (bin < 0 || bin > 3) { bin = 0; } /* any other RT3_BINNING: the unsorted kernel */
    ctx->stats_beam = beam; ctx->stats_beam_accel = beam_accel;
    const size_t smem = plan.smem + (bin ? RT3_BIN_SCRATCH_BYTES : 0) + (beam ? RT3_BEAM_BYTES : 0) + (beam_accel ? RT3_ABEAM_BYTES : 0);
    rc = beam_accel ? (bin == 3 ? launch_pathtrace<true, false, true, 3, true>(ctx, *cam, kp, smem, stream)
                                : launch_pathtrace<true, false, true, 0, true>(ctx, *cam, kp, smem, stream))
       : bin == 1 ? launch_pathtrace<true, false, true, 1>(ctx, *cam, kp, smem, stream)
       : bin == 2 ? launch_pathtrace<true, false, true, 2>(ctx, *cam, kp, smem, stream)
       : bin == 3 ? launch_pathtrace<true, false, true, 3>(ctx, *cam, kp, smem, stream)
       : beam ? launch_pathtrace<true, true, false, 0, true>(ctx, *cam, kp, smem, stream)
       : with_scene_variant(plan, [&](auto r, auto so, auto a) {
             return launch_pathtrace<decltype(r)::value, decltype(so)::value, decltype(a)::value>(ctx, *cam, kp, smem, stream);
         });
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_k1, stream));
    unsigned resolve_grid = (unsigned) ((kp.n_pixels + 255ull) / 256ull);
    resolve_kernel<<<resolve_grid, 256, 0, stream>>>(kp, ctx->accum.ptr, device_frame);
    RT3_CUDA(cudaGetLastError());
    RT3_CUDA(cudaEventRecord(ctx->ev_end, stream));
    ctx->stats.kernel_launches = accumulate ? 2 : 3;
    ctx->accum_kp = kp;
    ctx->accum_valid = true;
    if (!accumulate) { ctx->accum_cam = *cam; ctx->accum_cam_mixed = false; ctx->accum_first = kp.first_sample; }
    else if (memcmp(&ctx->accum_cam, cam, sizeof *cam) != 0) { ctx->accum_cam_mixed = true; }
    return RT3_OK;
}

int check_render_args(rt3_ctx* ctx, const rt3_camera* cam, const rt3_params* params, rt3_kparams* kp) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (!cam) { return fail(RT3_ERR_INVALID, "camera is NULL"); }
    if (!ctx->has_scene) { return fail(RT3_ERR_NO_SCENE, "rt3_scene_upload has not been called on this context"); }
    int rc = make_kparams(params, kp);
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    return RT3_OK;
}

/* Copies the rows this partition owns from the device frame to the host frame. */
template <class T>
int copy_owned_rows(const rt3_kparams& kp, const T* dev, T* host, cudaStream_t stream) {
    if (kp.part_count <= 1) {
        RT3_CUDA(cudaMemcpyAsync(host, dev, (size_t) kp.width * kp.height * sizeof(T), cudaMemcpyDeviceToHost, stream));
        return RT3_OK;
    }
    uint32_t n_tiles = (kp.height + kp.tile_rows - 1) / kp.tile_rows;
    for (uint32_t t = kp.part_index; t < n_tiles; t += kp.part_count) {
        uint32_t first = t * kp.tile_rows;
        uint32_t rows = (kp.height - first < kp.tile_rows) ? kp.height - first : kp.tile_rows;
        size_t off = (size_t) first * kp.width;
        RT3_CUDA(cudaMemcpyAsync(host + off, dev + off, (size_t) rows * kp.width * sizeof(T), cudaMemcpyDeviceToHost, stream));
    }
    return RT3_OK;
}

int collect_stats(rt3_ctx* ctx);

int render_to_host(rt3_ctx* ctx, const rt3_camera* cam, const rt3_params* params, uint32_t* host_frame, uint32_t* host_prim,
                   uint32_t* host_ent, float* host_t, bool want_aov) {
    rt3_kparams kp;
    int rc = check_render_args(ctx, cam, params, &kp);
    if (rc != RT3_OK) { return rc; }
    if (!host_frame) { return fail(RT3_ERR_INVALID, "host_frame is NULL"); }
    if (want_aov && params->mode != RT3_MODE_REFERENCE) { return fail(RT3_ERR_INVALID, "AOVs are only produced in RT3_MODE_REFERENCE"); }
    size_t n = (size_t) kp.width * kp.height;
    if ((rc = ctx->frame.reserve(n)) != RT3_OK) { return rc; }
    uint32_t *d_prim = nullptr, *d_ent = nullptr;
    float* d_t = nullptr;
    if (want_aov) {
        if (host_prim) { if ((rc = ctx->aov_prim.reserve(n)) != RT3_OK) { return rc; } d_prim = ctx->aov_prim.ptr; }
        if (host_ent) { if ((rc = ctx->aov_entity.reserve(n)) != RT3_OK) { return rc; } d_ent = ctx->aov_entity.ptr; }
        if (host_t) {
            ctx->path_aovs_valid = false; /* the depth buffer is the path-traced AOVs' too */
            if ((rc = ctx->aov_t.reserve(n)) != RT3_OK) { return rc; }
            d_t = ctx->aov_t.ptr;
        }
    }
    rc = enqueue_render(ctx, cam, params, kp, ctx->frame.ptr, d_prim, d_ent, d_t, ctx->stream);
    if (rc != RT3_OK) { return rc; }
    if ((rc = copy_owned_rows(kp, ctx->frame.ptr, host_frame, ctx->stream)) != RT3_OK) { return rc; }
    if (d_prim && (rc = copy_owned_rows(kp, d_prim, host_prim, ctx->stream)) != RT3_OK) { return rc; }
    if (d_ent && (rc = copy_owned_rows(kp, d_ent, host_ent, ctx->stream)) != RT3_OK) { return rc; }
    if (d_t && (rc = copy_owned_rows(kp, d_t, host_t, ctx->stream)) != RT3_OK) { return rc; }
    if ((rc = end_pass(ctx, ctx->stream)) != RT3_OK) { return rc; } /* blocking, like the reference's render() (VulkanRenderer.cpp:497) */
    if (ctx->stats.accel) { return collect_stats(ctx); } /* a traversal that overflowed its stack fails the render instead of dropping a subtree silently */
    return RT3_OK;
}

/* rt3_render_path_aovs: the AOV pass of the path tracer's primary rays on the context's stream, blocking. The sums live in
 * buffers of their own; the accumulators, accum_kp / accum_valid and the stream rt3_read_radiance orders itself behind are
 * left as they were. */
int render_path_aovs(rt3_ctx* ctx, const rt3_camera* cam, const rt3_params* params, const rt3_path_aovs* out) {
    if (!params || !out) { return fail(RT3_ERR_INVALID, "params or out is NULL"); }
    if (params->mode != RT3_MODE_PATHTRACE) { return fail(RT3_ERR_INVALID, "rt3_render_path_aovs takes RT3_MODE_PATHTRACE parameters only"); }
    rt3_params p = *params;
    p.max_depth = 1; /* ignored: primary rays only */
    p.flags &= RT3_FLAG_NO_JITTER | RT3_FLAG_UNIFORM_SKY | RT3_FLAG_BVH;
    rt3_kparams kp;
    int rc = check_render_args(ctx, cam, &p, &kp);
    if (rc != RT3_OK) { return rc; }
    const size_t n = (size_t) kp.width * kp.height;
    uint32_t *d_prim = nullptr, *d_ent = nullptr;
    ctx->path_aovs_valid = false;
    /* depth is kept on the device even when the caller does not want it: it guides rt3_denoise */
    if ((rc = ctx->aov_sums.reserve(RT3_AOV_SUMS * n)) != RT3_OK || (rc = ctx->aov_albedo.reserve(3 * n)) != RT3_OK ||
        (rc = ctx->aov_normal.reserve(3 * n)) != RT3_OK || (rc = ctx->aov_t.reserve(n)) != RT3_OK) {
        return rc;
    }
    float* d_t = ctx->aov_t.ptr;
    if (out->hit_prim) { if ((rc = ctx->aov_prim.reserve(n)) != RT3_OK) { return rc; } d_prim = ctx->aov_prim.ptr; }
    if (out->hit_entity) { if ((rc = ctx->aov_entity.reserve(n)) != RT3_OK) { return rc; } d_ent = ctx->aov_entity.ptr; }
    cudaStream_t stream = ctx->stream;
    trace_plan plan;
    if ((rc = plan_trace(ctx, p.flags, false, stream, &plan)) != RT3_OK) { return rc; }
    kp.resident = plan.resident ? 1u : 0u;
    cudaStream_t radiance_stream = ctx->last_stream;
    {
        std::unique_lock<std::mutex> bank_lock; /* held until the kernel that reads the bank is enqueued */
        if ((rc = begin_pass(ctx, plan.accel, kp.owned_rows, stream, plan.resident && kp.n_pixels != 0 ? &bank_lock : nullptr)) != RT3_OK) { return rc; }
        RT3_CUDA(cudaMemsetAsync(ctx->aov_sums.ptr, 0, RT3_AOV_SUMS * n * sizeof(unsigned long long), stream));
        RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
        if (kp.n_pixels != 0) {
            rc = with_scene_variant(plan, [&](auto r, auto so, auto a) {
                return launch_path_aovs<decltype(r)::value, decltype(so)::value, decltype(a)::value>(ctx, *cam, kp, plan.smem, d_prim, d_ent, d_t, stream);
            });
            if (rc != RT3_OK) { return rc; }
        }
    }
    RT3_CUDA(cudaEventRecord(ctx->ev_k1, stream));
    if (kp.n_pixels != 0) {
        path_aov_resolve_kernel<<<(unsigned) ((kp.n_pixels + 255ull) / 256ull), 256, 0, stream>>>(kp, ctx->aov_sums.ptr, ctx->aov_albedo.ptr, ctx->aov_normal.ptr);
        RT3_CUDA(cudaGetLastError());
        ctx->stats.kernel_launches = 2;
    }
    RT3_CUDA(cudaEventRecord(ctx->ev_end, stream));
    if (d_prim && (rc = copy_owned_rows(kp, d_prim, out->hit_prim, stream)) != RT3_OK) { return rc; }
    if (d_ent && (rc = copy_owned_rows(kp, d_ent, out->hit_entity, stream)) != RT3_OK) { return rc; }
    if (out->hit_t && (rc = copy_owned_rows(kp, d_t, out->hit_t, stream)) != RT3_OK) { return rc; }
    /* three floats per pixel: rows of float3 */
    if (out->albedo && (rc = copy_owned_rows(kp, reinterpret_cast<const float3*>(ctx->aov_albedo.ptr), reinterpret_cast<float3*>(out->albedo), stream)) != RT3_OK) { return rc; }
    if (out->normal && (rc = copy_owned_rows(kp, reinterpret_cast<const float3*>(ctx->aov_normal.ptr), reinterpret_cast<float3*>(out->normal), stream)) != RT3_OK) { return rc; }
    if ((rc = end_pass(ctx, stream)) != RT3_OK) { return rc; }
    rc = collect_stats(ctx);
    if (radiance_stream) { ctx->last_stream = radiance_stream; } /* rt3_read_radiance stays behind the render that filled the accumulators */
    if (rc == RT3_OK) {
        ctx->path_aovs_valid = true;
        ctx->path_aovs_kp = kp;
        ctx->path_aovs_cam = *cam;
        ctx->path_aovs_scene_id = ctx->scene_id;
    }
    return rc;
}

/* The conditions rt3_denoise and the calls for frames rendered in parts share: valid parameters, a path-traced render of
 * the frame's size whose passes used one camera, and path AOVs of the same size, camera and scene upload. `parts`: a
 * partition is allowed, and then the AOVs must have the render's. `fn` names the call in the messages. */
int check_denoise_inputs(rt3_ctx* ctx, const rt3_denoise_params* params, const char* fn, bool parts) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (const char* why = rt3_dn_check_params(params)) { return fail(RT3_ERR_INVALID, "%s: %s", fn, why); }
    if (!ctx->accum_valid) { return fail(RT3_ERR_INVALID, "%s needs a path-traced render on this context", fn); }
    const rt3_kparams& kp = ctx->accum_kp;
    if (params->width != kp.width || params->height != kp.height) {
        return fail(RT3_ERR_INVALID, "%s: the last path-traced frame was %ux%u, not %ux%u", fn, kp.width, kp.height, params->width, params->height);
    }
    if (!parts && kp.part_count > 1) { return fail(RT3_ERR_INVALID, "%s: the path-traced render covers part %u of %u of the frame, not all of it", fn, kp.part_index, kp.part_count); }
    if (ctx->accum_cam_mixed) { return fail(RT3_ERR_INVALID, "%s: the accumulated render's passes used different cameras", fn); }
    if (!ctx->path_aovs_valid) { return fail(RT3_ERR_INVALID, "%s needs an rt3_render_path_aovs on this context (after any rt3_render_aov with hit_t)", fn); }
    const rt3_kparams& ak = ctx->path_aovs_kp;
    if (!parts && ak.part_count > 1) { return fail(RT3_ERR_INVALID, "%s: the AOVs cover part %u of %u of the frame, not all of it", fn, ak.part_index, ak.part_count); }
    if (ak.width != kp.width || ak.height != kp.height) {
        return fail(RT3_ERR_INVALID, "%s: the AOVs are %ux%u, the render %ux%u", fn, ak.width, ak.height, kp.width, kp.height);
    }
    if (parts && (ak.tile_rows != kp.tile_rows || ak.part_index != kp.part_index || ak.part_count != kp.part_count)) {
        return fail(RT3_ERR_INVALID, "%s: the AOVs' partition (tile_rows %u, part %u of %u) differs from the render's (%u, %u of %u)", fn, ak.tile_rows,
                    ak.part_index, ak.part_count, kp.tile_rows, kp.part_index, kp.part_count);
    }
    if (memcmp(&ctx->path_aovs_cam, &ctx->accum_cam, sizeof(rt3_camera)) != 0) { return fail(RT3_ERR_INVALID, "%s: the AOVs and the render used different cameras", fn); }
    if (!ctx->has_scene || ctx->path_aovs_scene_id != ctx->scene_id) { return fail(RT3_ERR_INVALID, "%s: the AOVs were rendered from another scene upload than the render", fn); }
    return RT3_OK;
}

dim3 denoise_grid(uint32_t w, uint32_t h) { return dim3((w + RT3_DN_BLOCK_X - 1) / RT3_DN_BLOCK_X, (h + RT3_DN_BLOCK_Y - 1) / RT3_DN_BLOCK_Y); }

/* The stream rt3_read_radiance and the denoise calls enqueue on: the one of the render that filled the accumulators. */
cudaStream_t accum_stream(const rt3_ctx* ctx) { return ctx->last_stream ? ctx->last_stream : ctx->stream; }

/* The end of every filtering call, after the caller enqueued its preparation and variance kernels into dn_col[0] (colour
 * and variance) and counted them: the `iterations` à-trous passes guided by `guide`, ping-ponging through dn_col, the last
 * remodulating by `albedo` into dn_frame and dn_rgb; then the copies of the history length (when `host_length` is not
 * NULL), the frame and rgb to the host. Ends the pass begun by the caller, blocking, and reads its statistics. */
int atrous_to_host(rt3_ctx* ctx, const rt3_denoise_params* params, const rt3_dn_guide* guide, const float* albedo, uint32_t* host_frame, float* host_rgb,
                   float* host_length, cudaStream_t stream) {
    const uint32_t w = params->width, h = params->height, n_pow = (uint32_t) params->sigma_normal;
    const size_t n = (size_t) w * h;
    const float sigma_l = params->sigma_luminance, sigma_z = params->sigma_depth;
    const dim3 block(RT3_DN_BLOCK_X, RT3_DN_BLOCK_Y), grid = denoise_grid(w, h);
    const bool gamma = !(ctx->accum_kp.flags & RT3_FLAG_NO_GAMMA);
    for (uint32_t i = 0; i < params->iterations; i++) {
        const rt3_dn_px* in = ctx->dn_col[i & 1u].ptr;
        rt3_dn_px* out = ctx->dn_col[(i + 1u) & 1u].ptr;
        if (i + 1u < params->iterations) {
            denoise_atrous_kernel<false><<<grid, block, 0, stream>>>(w, h, 1u << i, sigma_l, sigma_z, n_pow, in, guide, out, nullptr, gamma, nullptr, nullptr);
        } else {
            denoise_atrous_kernel<true><<<grid, block, 0, stream>>>(w, h, 1u << i, sigma_l, sigma_z, n_pow, in, guide, nullptr, albedo, gamma,
                                                                    ctx->dn_frame.ptr, host_rgb ? ctx->dn_rgb.ptr : nullptr);
        }
        RT3_CUDA(cudaGetLastError());
    }
    RT3_CUDA(cudaEventRecord(ctx->ev_k1, stream));
    RT3_CUDA(cudaEventRecord(ctx->ev_end, stream));
    ctx->stats.kernel_launches += params->iterations;
    if (host_length) { RT3_CUDA(cudaMemcpyAsync(host_length, ctx->dn_hist_length.ptr, n * sizeof(float), cudaMemcpyDeviceToHost, stream)); }
    if (host_frame) { RT3_CUDA(cudaMemcpyAsync(host_frame, ctx->dn_frame.ptr, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream)); }
    if (host_rgb) { RT3_CUDA(cudaMemcpyAsync(host_rgb, ctx->dn_rgb.ptr, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, stream)); }
    int rc = end_pass(ctx, stream);
    if (rc != RT3_OK) { return rc; }
    return collect_stats(ctx);
}

/* The filter's ping-pong buffers and outputs (plus the guides when `guide`), sized on first use. */
int reserve_denoise(rt3_ctx* ctx, size_t n, bool guide, bool rgb) {
    int rc;
    if ((rc = ctx->dn_col[0].reserve(n)) != RT3_OK || (rc = ctx->dn_col[1].reserve(n)) != RT3_OK || (guide && (rc = ctx->dn_guide.reserve(n)) != RT3_OK) ||
        (rc = ctx->dn_frame.reserve(n)) != RT3_OK || (rgb && (rc = ctx->dn_rgb.reserve(3 * n)) != RT3_OK)) {
        return rc;
    }
    return RT3_OK;
}

/* rt3_denoise: prepare, variance and `iterations` à-trous passes over the accumulators and the path-traced AOVs, on the
 * stream rt3_read_radiance orders itself behind (the one of the render that filled the accumulators), blocking. Reads the
 * accumulators and the AOV buffers and writes only the dn_* buffers; every condition is checked before anything changes. */
int denoise(rt3_ctx* ctx, const rt3_denoise_params* params, uint32_t* host_frame, float* host_rgb) {
    int rc = check_denoise_inputs(ctx, params, "rt3_denoise", false);
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const rt3_kparams& kp = ctx->accum_kp;
    const size_t n = (size_t) kp.width * kp.height;
    if ((rc = reserve_denoise(ctx, n, true, host_rgb != nullptr)) != RT3_OK) { return rc; }
    cudaStream_t stream = accum_stream(ctx);
    if ((rc = begin_pass(ctx, false, kp.height, stream, nullptr)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
    denoise_prepare_kernel<<<(unsigned) ((n + 255) / 256), 256, 0, stream>>>(kp, ctx->accum.ptr, ctx->aov_albedo.ptr, ctx->aov_normal.ptr, ctx->aov_t.ptr,
                                                                           ctx->dn_col[1].ptr, ctx->dn_guide.ptr);
    RT3_CUDA(cudaGetLastError());
    denoise_variance_kernel<<<denoise_grid(kp.width, kp.height), dim3(RT3_DN_BLOCK_X, RT3_DN_BLOCK_Y), 0, stream>>>(
        kp.width, kp.height, params->sigma_depth, (uint32_t) params->sigma_normal, ctx->dn_col[1].ptr, ctx->dn_guide.ptr, ctx->dn_col[0].ptr);
    RT3_CUDA(cudaGetLastError());
    ctx->stats.kernel_launches += 2;
    return atrous_to_host(ctx, params, ctx->dn_guide.ptr, ctx->aov_albedo.ptr, host_frame, host_rgb, nullptr, stream);
}

/* The start of a temporal call (rt3_denoise_temporal, rt3_denoise_staged_temporal), after every check: whether the
 * history may be read (*have_prev: not reset, and one of this size and scene upload), then drops it until keep_history
 * and sizes both histories (and the length for the host when `length`) and the filter's buffers (reserve_denoise). */
int begin_history(rt3_ctx* ctx, const rt3_denoise_temporal_params* tp, uint32_t w, uint32_t h, bool guide, bool rgb, bool length, bool* have_prev) {
    const size_t n = (size_t) w * h;
    *have_prev = !tp->reset && ctx->dn_hist_valid && ctx->dn_hist_width == w && ctx->dn_hist_height == h && ctx->dn_hist_scene_id == ctx->scene_id;
    ctx->dn_hist_valid = false;
    int rc;
    if ((rc = reserve_denoise(ctx, n, guide, rgb)) != RT3_OK) { return rc; }
    for (uint32_t i = 0; i < 2; i++) {
        if ((rc = ctx->dn_hist_col[i].reserve(n)) != RT3_OK || (rc = ctx->dn_hist_mom[i].reserve(n)) != RT3_OK || (rc = ctx->dn_hist_guide[i].reserve(n)) != RT3_OK) {
            return rc;
        }
    }
    if (length && (rc = ctx->dn_hist_length.reserve(n)) != RT3_OK) { return rc; }
    return RT3_OK;
}

/* The end of a temporal call that succeeded: the history it wrote becomes the one the next call reads, with the AOVs'
 * camera, the frame's size and the scene upload. */
void keep_history(rt3_ctx* ctx, uint32_t w, uint32_t h) {
    ctx->dn_hist_cur ^= 1u;
    ctx->dn_hist_valid = true;
    ctx->dn_hist_cam = ctx->path_aovs_cam;
    ctx->dn_hist_width = w; ctx->dn_hist_height = h;
    ctx->dn_hist_scene_id = ctx->scene_id;
}

/* rt3_denoise_temporal: rt3_denoise's checks and the temporal parameters', then the accumulation into the history not in
 * use, its variance, the à-trous passes and the read-back, blocking. The history is dropped when the call proceeds and
 * kept (swapped in) only when everything succeeded; a refusal changes nothing. */
int denoise_temporal(rt3_ctx* ctx, const rt3_denoise_temporal_params* tp, uint32_t* host_frame, float* host_rgb, float* host_length) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (!tp) { return fail(RT3_ERR_INVALID, "rt3_denoise_temporal: params is NULL"); }
    int rc = check_denoise_inputs(ctx, &tp->filter, "rt3_denoise_temporal", false);
    if (rc != RT3_OK) { return rc; }
    if (const char* why = rt3_dn_check_temporal_params(tp)) { return fail(RT3_ERR_INVALID, "rt3_denoise_temporal: %s", why); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const rt3_kparams& kp = ctx->accum_kp;
    const uint32_t w = kp.width, h = kp.height;
    bool have_prev;
    if ((rc = begin_history(ctx, tp, w, h, true, host_rgb != nullptr, host_length != nullptr, &have_prev)) != RT3_OK) { return rc; }
    const uint32_t cur = ctx->dn_hist_cur, next = cur ^ 1u;
    cudaStream_t stream = accum_stream(ctx);
    if ((rc = begin_pass(ctx, false, h, stream, nullptr)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
    const dim3 block(RT3_DN_BLOCK_X, RT3_DN_BLOCK_Y), grid = denoise_grid(w, h);
    denoise_temporal_kernel<<<grid, block, 0, stream>>>(kp, ctx->path_aovs_kp, ctx->path_aovs_cam, ctx->dn_hist_cam, *tp, have_prev, ctx->accum.ptr,
                                                        ctx->aov_albedo.ptr, ctx->aov_normal.ptr, ctx->aov_t.ptr, ctx->dn_hist_col[cur].ptr,
                                                        ctx->dn_hist_mom[cur].ptr, ctx->dn_hist_guide[cur].ptr, ctx->dn_hist_col[next].ptr,
                                                        ctx->dn_hist_mom[next].ptr, ctx->dn_hist_guide[next].ptr, ctx->dn_col[1].ptr, ctx->dn_guide.ptr,
                                                        host_length ? ctx->dn_hist_length.ptr : nullptr);
    RT3_CUDA(cudaGetLastError());
    const rt3_denoise_params& fp = tp->filter;
    denoise_temporal_variance_kernel<<<grid, block, 0, stream>>>(w, h, fp.sigma_depth, (uint32_t) fp.sigma_normal, ctx->dn_col[1].ptr, ctx->dn_guide.ptr,
                                                                 ctx->dn_hist_col[next].ptr, ctx->dn_hist_mom[next].ptr, ctx->dn_col[0].ptr);
    RT3_CUDA(cudaGetLastError());
    ctx->stats.kernel_launches += 2;
    if ((rc = atrous_to_host(ctx, &fp, ctx->dn_guide.ptr, ctx->aov_albedo.ptr, host_frame, host_rgb, host_length, stream)) != RT3_OK) { return rc; }
    keep_history(ctx, w, h);
    return RT3_OK;
}

/* Where the planes of a stage of rt3_denoise_stage_words(w, h) words start (include/rt3cuda.h). */
struct stage_view {
    rt3_dn_px* col;
    rt3_dn_guide* guide;
    float* albedo;
    unsigned long long* fingerprint;
};

uint64_t stage_fingerprint_offset(uint64_t n) { return (11ull * n + 1ull) & ~1ull; }

stage_view stage_planes(uint32_t* stage, uint32_t w, uint32_t h) {
    const uint64_t n = (uint64_t) w * h;
    return { reinterpret_cast<rt3_dn_px*>(stage), reinterpret_cast<rt3_dn_guide*>(stage + 4 * n), reinterpret_cast<float*>(stage + 8 * n),
             reinterpret_cast<unsigned long long*>(stage + stage_fingerprint_offset(n)) };
}

uint64_t fnv1a(uint64_t hash, const void* data, size_t bytes) {
    const unsigned char* b = static_cast<const unsigned char*>(data);
    for (size_t i = 0; i < bytes; i++) { hash = (hash ^ b[i]) * 0x100000001b3ull; }
    return hash;
}

/* The rows' fingerprint for this context's render and AOVs (include/rt3cuda.h): nonzero, and equal on two parts exactly
 * when their filter inputs are pixels of the same frame. */
uint64_t stage_fingerprint(const rt3_ctx* ctx, uint64_t frame_tag) {
    const rt3_kparams& kp = ctx->accum_kp;
    const rt3_kparams& ak = ctx->path_aovs_kp;
    const uint32_t sampling = RT3_FLAG_NO_JITTER | RT3_FLAG_UNIFORM_SKY;
    const uint32_t fields[] = { kp.width, kp.height, kp.seed, kp.max_depth, ctx->accum_first, kp.first_sample + kp.spp, kp.resolve_spp,
                                kp.flags & (sampling | RT3_FLAG_NO_GAMMA), kp.tile_rows, kp.part_count, ak.seed, ak.spp, ak.first_sample, ak.flags & sampling };
    uint64_t hash = fnv1a(0xcbf29ce484222325ull, &frame_tag, sizeof frame_tag);
    hash = fnv1a(hash, fields, sizeof fields);
    hash = fnv1a(hash, &ctx->accum_cam, sizeof(rt3_camera));
    return hash ? hash : 1ull;
}

/* rt3_denoise_stage: denoise_stage_kernel over the owned rows, asynchronous on `stream`; rt3_get_stats waits for it. */
int denoise_stage(rt3_ctx* ctx, const rt3_denoise_params* params, uint64_t frame_tag, uint32_t* device_stage, cudaStream_t user_stream) {
    int rc = check_denoise_inputs(ctx, params, "rt3_denoise_stage", true);
    if (rc != RT3_OK) { return rc; }
    if (!device_stage) { return fail(RT3_ERR_INVALID, "rt3_denoise_stage: device_stage is NULL"); }
    const rt3_kparams& kp = ctx->accum_kp;
    if (rt3_denoise_stage_words(kp.width, kp.height) == 0) { return fail(RT3_ERR_INVALID, "rt3_denoise_stage: a %ux%u frame does not fit in a stage", kp.width, kp.height); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t stream = user_stream ? user_stream : accum_stream(ctx);
    const stage_view s = stage_planes(device_stage, kp.width, kp.height);
    if ((rc = begin_pass(ctx, false, kp.owned_rows, stream, nullptr)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
    if (kp.n_pixels != 0) {
        denoise_stage_kernel<<<(unsigned) ((kp.n_pixels + 255ull) / 256ull), 256, 0, stream>>>(kp, ctx->accum.ptr, ctx->aov_albedo.ptr, ctx->aov_normal.ptr,
                                                                                              ctx->aov_t.ptr, s.col, s.guide, s.albedo, s.fingerprint,
                                                                                              stage_fingerprint(ctx, frame_tag));
        RT3_CUDA(cudaGetLastError());
        ctx->stats.kernel_launches = 1;
    }
    RT3_CUDA(cudaEventRecord(ctx->ev_k1, stream));
    RT3_CUDA(cudaEventRecord(ctx->ev_end, stream));
    return RT3_OK;
}

/* The checks of the owner's calls on a stage (rt3_denoise_staged, rt3_denoise_staged_temporal, named by `fn`), after
 * check_denoise_inputs: a stage, a frame that fits one, and every row's fingerprint equal to this context's for frame_tag,
 * read back on `stream` (blocking). Sets the device and *s, the stage's planes. */
int check_stage_rows(rt3_ctx* ctx, const char* fn, uint64_t frame_tag, const uint32_t* device_stage, cudaStream_t stream, stage_view* s) {
    if (!device_stage) { return fail(RT3_ERR_INVALID, "%s: device_stage is NULL", fn); }
    const uint32_t w = ctx->accum_kp.width, h = ctx->accum_kp.height;
    if (rt3_denoise_stage_words(w, h) == 0) { return fail(RT3_ERR_INVALID, "%s: a %ux%u frame does not fit in a stage", fn, w, h); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    *s = stage_planes(const_cast<uint32_t*>(device_stage), w, h);
    std::vector<unsigned long long> rows(h);
    RT3_CUDA(cudaMemcpyAsync(rows.data(), s->fingerprint, h * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
    RT3_CUDA(cudaStreamSynchronize(stream));
    const unsigned long long expect = stage_fingerprint(ctx, frame_tag);
    uint32_t bad = 0, first_bad = 0;
    for (uint32_t y = 0; y < h; y++) {
        if (rows[y] != expect && bad++ == 0) { first_bad = y; }
    }
    if (bad) {
        return fail(RT3_ERR_INVALID, "%s: row %u (and %u rows in all, of %u) was not staged for this frame: a part that did not run, a stale row of "
                    "another frame_tag, or a part rendered with other parameters", fn, first_bad, bad, h);
    }
    return RT3_OK;
}

/* rt3_denoise_staged: checks every row's fingerprint on the host, then the filter over the stage's planes, blocking. */
int denoise_staged(rt3_ctx* ctx, const rt3_denoise_params* params, uint64_t frame_tag, const uint32_t* device_stage, uint32_t* host_frame, float* host_rgb) {
    int rc = check_denoise_inputs(ctx, params, "rt3_denoise_staged", true);
    if (rc != RT3_OK) { return rc; }
    const rt3_kparams& kp = ctx->accum_kp;
    const uint32_t w = kp.width, h = kp.height;
    cudaStream_t stream = accum_stream(ctx);
    stage_view s;
    if ((rc = check_stage_rows(ctx, "rt3_denoise_staged", frame_tag, device_stage, stream, &s)) != RT3_OK) { return rc; }
    if ((rc = reserve_denoise(ctx, (size_t) w * h, false, host_rgb != nullptr)) != RT3_OK) { return rc; }
    if ((rc = begin_pass(ctx, false, h, stream, nullptr)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
    denoise_variance_kernel<<<denoise_grid(w, h), dim3(RT3_DN_BLOCK_X, RT3_DN_BLOCK_Y), 0, stream>>>(w, h, params->sigma_depth, (uint32_t) params->sigma_normal,
                                                                                                   s.col, s.guide, ctx->dn_col[0].ptr);
    RT3_CUDA(cudaGetLastError());
    ctx->stats.kernel_launches += 1;
    return atrous_to_host(ctx, params, s.guide, s.albedo, host_frame, host_rgb, nullptr, stream);
}

/* rt3_denoise_staged_temporal: rt3_denoise_staged's checks and the temporal parameters', then rt3_denoise_temporal's
 * steps on the owner's history with the pixels read from the stage, blocking. The rays are regenerated from the owner's
 * AOV kparams with the partition removed: every part traced its rows with the same seed, sample range, flags and camera
 * (the fingerprints), and start_path then takes the pixel index. */
int denoise_staged_temporal(rt3_ctx* ctx, const rt3_denoise_temporal_params* tp, uint64_t frame_tag, const uint32_t* device_stage, uint32_t* host_frame,
                            float* host_rgb, float* host_length) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (!tp) { return fail(RT3_ERR_INVALID, "rt3_denoise_staged_temporal: params is NULL"); }
    int rc = check_denoise_inputs(ctx, &tp->filter, "rt3_denoise_staged_temporal", true);
    if (rc != RT3_OK) { return rc; }
    if (const char* why = rt3_dn_check_temporal_params(tp)) { return fail(RT3_ERR_INVALID, "rt3_denoise_staged_temporal: %s", why); }
    const uint32_t w = ctx->accum_kp.width, h = ctx->accum_kp.height;
    cudaStream_t stream = accum_stream(ctx);
    stage_view s;
    if ((rc = check_stage_rows(ctx, "rt3_denoise_staged_temporal", frame_tag, device_stage, stream, &s)) != RT3_OK) { return rc; }
    bool have_prev;
    if ((rc = begin_history(ctx, tp, w, h, false, host_rgb != nullptr, host_length != nullptr, &have_prev)) != RT3_OK) { return rc; }
    const uint32_t cur = ctx->dn_hist_cur, next = cur ^ 1u;
    rt3_kparams whole = ctx->path_aovs_kp;
    whole.part_index = 0; whole.part_count = 1; whole.owned_rows = h;
    whole.n_pixels = (unsigned long long) w * h;
    whole.n_items = whole.n_pixels * whole.spp;
    if ((rc = begin_pass(ctx, false, h, stream, nullptr)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ctx->ev_k0, stream));
    const dim3 block(RT3_DN_BLOCK_X, RT3_DN_BLOCK_Y), grid = denoise_grid(w, h);
    denoise_staged_temporal_kernel<<<grid, block, 0, stream>>>(whole, ctx->path_aovs_cam, ctx->dn_hist_cam, *tp, have_prev, s.col, s.guide,
                                                               ctx->dn_hist_col[cur].ptr, ctx->dn_hist_mom[cur].ptr, ctx->dn_hist_guide[cur].ptr,
                                                               ctx->dn_hist_col[next].ptr, ctx->dn_hist_mom[next].ptr, ctx->dn_hist_guide[next].ptr,
                                                               ctx->dn_col[1].ptr, host_length ? ctx->dn_hist_length.ptr : nullptr);
    RT3_CUDA(cudaGetLastError());
    const rt3_denoise_params& fp = tp->filter;
    denoise_temporal_variance_kernel<<<grid, block, 0, stream>>>(w, h, fp.sigma_depth, (uint32_t) fp.sigma_normal, ctx->dn_col[1].ptr, s.guide,
                                                                 ctx->dn_hist_col[next].ptr, ctx->dn_hist_mom[next].ptr, ctx->dn_col[0].ptr);
    RT3_CUDA(cudaGetLastError());
    ctx->stats.kernel_launches += 2;
    if ((rc = atrous_to_host(ctx, &fp, s.guide, s.albedo, host_frame, host_rgb, host_length, stream)) != RT3_OK) { return rc; }
    keep_history(ctx, w, h);
    return RT3_OK;
}

/* Reads back the timings and counters of the most recent render (synchronises its stream). */
int collect_stats(rt3_ctx* ctx) {
    if (!ctx->stats_pending) { return RT3_OK; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaStreamSynchronize(ctx->last_stream));
    unsigned long long counters[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    RT3_CUDA(cudaMemcpy(counters, ctx->counters.ptr, sizeof counters, cudaMemcpyDeviceToHost));
    float ms = 0.0f, ms_k = 0.0f, ms_copy = 0.0f;
    RT3_CUDA(cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
    RT3_CUDA(cudaEventElapsedTime(&ms_k, ctx->ev_k0, ctx->ev_k1));
    if (ctx->copy_timed) { RT3_CUDA(cudaEventElapsedTime(&ms_copy, ctx->ev_end, ctx->ev_copy)); }
    ctx->stats.device_ms = ms;
    ctx->stats.trace_kernel_ms = ms_k;
    ctx->stats.h2d_ms = 0.0;
    ctx->stats.d2h_ms = ms_copy;
    ctx->stats.rays = counters[1];
    ctx->stats.sphere_tests = counters[1] * ctx->view.n_spheres;
    ctx->stats.face_tests = counters[1] * ctx->view.n_faces;
    ctx->stats.beam_rays = 0; ctx->stats.beam_tests = 0;
    if (ctx->stats_beam && !ctx->stats.accel) {
        /* primary rays that were traced against their chunk's candidate list did not sweep the scene: they ran beam_tests exact tests */
        ctx->stats.beam_rays = counters[2]; ctx->stats.beam_tests = counters[3];
        ctx->stats.sphere_tests = (counters[1] - counters[2]) * ctx->view.n_spheres + counters[3];
    }
    if (ctx->stats.accel) {
        /* through the hierarchy only the leaves reached are tested */
        ctx->stats.sphere_tests = 0; ctx->stats.face_tests = 0;
    }
    if (ctx->stats.accel && ctx->stats_beam_accel) { ctx->stats.beam_rays = counters[5]; ctx->stats.beam_tests = counters[6]; }
    ctx->stats.accel_node_visits = ctx->stats.accel ? counters[2] : 0;
    ctx->stats.accel_prim_tests = ctx->stats.accel ? counters[3] : 0;
    ctx->stats.accel_build_ms = ctx->bvh_build_ms;
    ctx->stats.accel_stack_overflows = (uint32_t) std::min<unsigned long long>(counters[4], 0xFFFFFFFFull);
    ctx->stats_pending = false;
    if (counters[4]) { return fail(RT3_ERR_INVALID, "hierarchy traversal overflowed its stack %llu times: the frame may miss hits", counters[4]); }
    return RT3_OK;
}

int check_scene_args(const rt3_scene* s) {
    if (s->n_faces && (!s->faces || !s->vertices)) { return fail(RT3_ERR_INVALID, "faces/vertices missing"); }
    if (s->n_spheres && !s->spheres) { return fail(RT3_ERR_INVALID, "spheres missing"); }
    if ((s->face_material || s->sphere_material) && s->n_materials && !s->materials) { return fail(RT3_ERR_INVALID, "materials missing"); }
    if ((unsigned long long) s->n_faces + s->n_spheres > 0x7FFFFFFFull) { return fail(RT3_ERR_INVALID, "too many primitives"); }
    return RT3_OK;
}

/* Copies one host input array into a scratch device buffer as it is and points *device_view at it (NULL stays NULL). */
template <class T> int stage(DeviceBuffer<unsigned char>& buf, const T* host, size_t bytes, const T** device_view, cudaStream_t stream) {
    if (!host || bytes == 0) { *device_view = nullptr; return RT3_OK; }
    int rc = buf.reserve(bytes);
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaMemcpyAsync(buf.ptr, host, bytes, cudaMemcpyHostToDevice, stream));
    *device_view = reinterpret_cast<const T*>(buf.ptr);
    return RT3_OK;
}

__global__ void build_init_kernel(rt3_build_info* info) {
    info->error_key = ~0ull; info->n_valid = 0ull; info->ray_slack = 0.f; info->r2_median = 1.0; info->r2_min = 1.0;
    for (int k = 0; k < 4; k++) { info->error_detail[k] = 0u; }
    for (int k = 0; k < 3; k++) { info->cmin_bits[k] = 0x7fffffff; info->cmax_bits[k] = (int) 0x80000000; }
}

/* Every derived scene array from flattened inputs that lie in device memory (`d` holds device pointers): the
 * kernels of rt3_upload.cuh on the context's stream, one small read-back (validation result, basis, slack,
 * centroid box) at the end. Replaces any previous scene of the context. */
int build_scene_on_device(rt3_ctx* ctx, const rt3_scene& d) {
    cudaStream_t stream = ctx->stream;
    ctx->has_scene = false;
    ctx->accum_valid = false; /* the accumulators belong to the previous scene */
    ctx->bvh_ready = false;
    const uint32_t nf = d.n_faces, ns = d.n_spheres, np = nf + ns;
    const uint32_t np_pad = (np + RT3_PAD_PRIMS - 1) / RT3_PAD_PRIMS * RT3_PAD_PRIMS;
    int rc;
    auto at_least_one = [](size_t n) { return n ? n : (size_t) 1; };
    if ((rc = ctx->face_rec.reserve(at_least_one(4 * (size_t) nf))) != RT3_OK ||
        (rc = ctx->spheres.reserve(at_least_one(ns))) != RT3_OK || (rc = ctx->prim_color.reserve(at_least_one(np))) != RT3_OK ||
        (rc = ctx->prim_material.reserve(at_least_one(np))) != RT3_OK || (rc = ctx->prim_entity.reserve(at_least_one(np))) != RT3_OK ||
        (rc = ctx->prim_lo.reserve(at_least_one(np))) != RT3_OK || (rc = ctx->prim_hi.reserve(at_least_one(np))) != RT3_OK ||
        (rc = ctx->filt3.reserve(at_least_one(np_pad))) != RT3_OK || (rc = ctx->pair_xy.reserve(at_least_one(np_pad / 2))) != RT3_OK ||
        (rc = ctx->pair_w.reserve(at_least_one(np_pad / 2))) != RT3_OK || (rc = ctx->materials.reserve(at_least_one((size_t) d.n_materials * 2))) != RT3_OK) {
        return rc;
    }
    DeviceBuffer<rt3_bound> bounds;
    DeviceBuffer<float> keys_in, keys_out;
    DeviceBuffer<double> partials;
    DeviceBuffer<rt3_build_info> info;
    DeviceBuffer<unsigned char> temp;
    if ((rc = bounds.reserve(at_least_one(np))) != RT3_OK || (rc = keys_in.reserve(at_least_one(np))) != RT3_OK || (rc = keys_out.reserve(at_least_one(np))) != RT3_OK ||
        (rc = partials.reserve(RT3_MOMENT_BLOCKS * RT3_MOMENTS)) != RT3_OK || (rc = info.reserve(1)) != RT3_OK) {
        return rc;
    }
    size_t temp_bytes = 0;
    if (np) { RT3_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, temp_bytes, keys_in.ptr, keys_out.ptr, (int) np, 0, 32, stream)); }
    if ((rc = temp.reserve(at_least_one(temp_bytes))) != RT3_OK) { return rc; }
    EventPair ev;
    if ((rc = ev.create()) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ev.begin, stream));
    build_init_kernel<<<1, 1, 0, stream>>>(info.ptr);
    RT3_CUDA(cudaGetLastError());
    rt3_build_out out;
    out.face_rec = ctx->face_rec.ptr;
    out.spheres = ctx->spheres.ptr; out.prim_color = ctx->prim_color.ptr; out.prim_lo = ctx->prim_lo.ptr; out.prim_hi = ctx->prim_hi.ptr;
    out.prim_material = ctx->prim_material.ptr; out.prim_entity = ctx->prim_entity.ptr; out.bounds = bounds.ptr; out.r2_keys = keys_in.ptr;
    if (nf) {
        build_faces_kernel<<<(nf + 255u) / 256u, 256, 0, stream>>>(nf, d.n_vertices, reinterpret_cast<const uint4*>(d.faces), reinterpret_cast<const float4*>(d.vertices),
                                                                     d.face_material, d.face_entity, d.n_materials, out, info.ptr);
        RT3_CUDA(cudaGetLastError());
    }
    if (ns) {
        build_spheres_kernel<<<(ns + 255u) / 256u, 256, 0, stream>>>(nf, ns, reinterpret_cast<const float4*>(d.spheres), d.sphere_color, d.sphere_material,
                                                                       d.sphere_entity, d.n_materials, out, info.ptr);
        RT3_CUDA(cudaGetLastError());
    }
    if (d.n_materials && d.materials) {
        build_materials_kernel<<<(d.n_materials + 255u) / 256u, 256, 0, stream>>>(d.n_materials, reinterpret_cast<const uint4*>(d.materials), ctx->materials.ptr, info.ptr);
        RT3_CUDA(cudaGetLastError());
    }
    if (np) {
        size_t tb = temp_bytes;
        RT3_CUDA(cub::DeviceRadixSort::SortKeys(temp.ptr, tb, keys_in.ptr, keys_out.ptr, (int) np, 0, 32, stream));
    }
    build_radius_stats_kernel<<<1, 1, 0, stream>>>(keys_out.ptr, info.ptr);
    RT3_CUDA(cudaGetLastError());
    build_moments_kernel<<<RT3_MOMENT_BLOCKS, RT3_MOMENT_THREADS, 0, stream>>>(np, bounds.ptr, info.ptr, partials.ptr);
    RT3_CUDA(cudaGetLastError());
    build_basis_kernel<<<1, 1, 0, stream>>>(partials.ptr, info.ptr);
    RT3_CUDA(cudaGetLastError());
    if (np_pad) {
        build_records_kernel<<<(np_pad / 2 + 255u) / 256u, 256, 0, stream>>>(np, np_pad / 2, bounds.ptr, ctx->prim_lo.ptr, ctx->prim_hi.ptr, ctx->filt3.ptr,
                                                                              ctx->pair_xy.ptr, ctx->pair_w.ptr, info.ptr);
        RT3_CUDA(cudaGetLastError());
    }
    RT3_CUDA(cudaEventRecord(ev.end, stream));
    rt3_build_info h;
    RT3_CUDA(cudaMemcpyAsync(&h, info.ptr, sizeof h, cudaMemcpyDeviceToHost, stream));
    RT3_CUDA(cudaStreamSynchronize(stream)); /* also: the scratch arrays (and the caller's staging buffers) go out of scope */
    float ms = 0.f;
    RT3_CUDA(cudaEventElapsedTime(&ms, ev.begin, ev.end));
    ctx->upload_device_ms = ms;
    if (h.error_key != ~0ull) {
        const unsigned stage_id = (unsigned) (h.error_key >> 62), kind = (unsigned) (h.error_key & 3ull);
        const uint32_t index = (uint32_t) ((h.error_key >> 2) & 0xFFFFFFFFull);
        if (kind == RT3_BUILD_ERR_VERTEX) {
            return fail(RT3_ERR_INVALID, "face %u references vertex out of range (%u,%u,%u of %u)", index, h.error_detail[0], h.error_detail[1], h.error_detail[2], h.error_detail[3]);
        }
        if (kind == RT3_BUILD_ERR_MATERIAL) { return fail(RT3_ERR_INVALID, "%s %u: material %u out of range", stage_id == 0 ? "face" : "sphere", index, h.error_detail[0]); }
        return fail(RT3_ERR_INVALID, "material %u: unknown kind %u", index, h.error_detail[0]);
    }
    for (int k = 0; k < 3; k++) {
        float lo = ordered_to_float(h.cmin_bits[k]), hi = ordered_to_float(h.cmax_bits[k]);
        if (!(lo <= hi)) { lo = hi = 0.0f; }
        ctx->centroid_min[k] = lo; ctx->centroid_max[k] = hi;
    }
    rt3_scene_view& v = ctx->view;
    for (int k = 0; k < 3; k++) { v.e1[k] = h.basis[0][k]; v.e2[k] = h.basis[1][k]; v.e3[k] = h.basis[2][k]; }
    v.ray_slack = h.ray_slack;
    ctx->scene_id = g_next_scene_id.fetch_add(1);
    v.n_faces = nf; v.n_spheres = ns; v.n_prims = np; v.n_prims_padded = np_pad;
    v.pair_xy = ctx->pair_xy.ptr; v.pair_w = ctx->pair_w.ptr; v.filt3 = ctx->filt3.ptr;
    v.face_rec = ctx->face_rec.ptr;
    v.spheres = ctx->spheres.ptr; v.prim_color = ctx->prim_color.ptr;
    v.prim_material = ctx->prim_material.ptr; v.prim_entity = ctx->prim_entity.ptr; v.materials = ctx->materials.ptr;
    ctx->has_scene = true;
    return RT3_OK;
}

}  // namespace

extern "C" {

const char* rt3_last_error(void) { return g_error.c_str(); }

int rt3_create(rt3_ctx** out, int device) {
    if (!out) { return fail(RT3_ERR_INVALID, "out is NULL"); }
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        return fail(RT3_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= n_dev || device >= RT3_MAX_DEVICES) { return fail(RT3_ERR_INVALID, "device %d out of range (0..%d)", device, std::min(n_dev, RT3_MAX_DEVICES) - 1); }
    RT3_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RT3_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { return fail(RT3_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); }
    rt3_ctx* ctx = new rt3_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    cudaError_t err = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (err == cudaSuccess) { err = cudaEventCreate(&ctx->ev_begin); }
    if (err == cudaSuccess) { err = cudaEventCreate(&ctx->ev_end); }
    if (err == cudaSuccess) { err = cudaEventCreate(&ctx->ev_copy); }
    if (err == cudaSuccess) { err = cudaEventCreate(&ctx->ev_k0); }
    if (err == cudaSuccess) { err = cudaEventCreate(&ctx->ev_k1); }
    if (err == cudaSuccess && ctx->counters.reserve(8) != RT3_OK) { err = cudaErrorMemoryAllocation; }
    if (err != cudaSuccess) {
        rt3_destroy(ctx);
        return fail(RT3_ERR_CUDA, "context setup failed: %s", cudaGetErrorString(err));
    }
    *out = ctx;
    return RT3_OK;
}

int rt3_destroy(rt3_ctx* ctx) {
    if (!ctx) { return RT3_OK; }
    cudaSetDevice(ctx->device);
    if (ctx->stream) { cudaStreamSynchronize(ctx->stream); }
    if (ctx->ev_begin) { cudaEventDestroy(ctx->ev_begin); }
    if (ctx->ev_end) { cudaEventDestroy(ctx->ev_end); }
    if (ctx->ev_copy) { cudaEventDestroy(ctx->ev_copy); }
    if (ctx->ev_k0) { cudaEventDestroy(ctx->ev_k0); }
    if (ctx->ev_k1) { cudaEventDestroy(ctx->ev_k1); }
    if (ctx->stream) { cudaStreamDestroy(ctx->stream); }
    delete ctx;
    return RT3_OK;
}

int rt3_scene_upload(rt3_ctx* ctx, const rt3_scene* s) {
    if (!ctx || !s) { return fail(RT3_ERR_INVALID, "ctx or scene is NULL"); }
    int rc = check_scene_args(s);
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const auto t0 = std::chrono::steady_clock::now();
    /* stage the flattened arrays as they are (one copy per array, nothing per primitive on the host); every derived
     * array is then built by kernels (rt3_upload.cuh) */
    DeviceBuffer<unsigned char> faces, vertices, face_material, face_entity, spheres, sphere_color, sphere_material, sphere_entity, materials;
    rt3_scene d = *s;
    EventPair ev;
    if ((rc = ev.create()) != RT3_OK) { return rc; }
    RT3_CUDA(cudaEventRecord(ev.begin, ctx->stream));
    if ((rc = stage(faces, s->faces, (size_t) s->n_faces * sizeof(rt3_face), &d.faces, ctx->stream)) != RT3_OK ||
        (rc = stage(vertices, s->vertices, (size_t) s->n_vertices * sizeof(rt3_vertex), &d.vertices, ctx->stream)) != RT3_OK ||
        (rc = stage(face_material, s->face_material, (size_t) s->n_faces * 4, &d.face_material, ctx->stream)) != RT3_OK ||
        (rc = stage(face_entity, s->face_entity, (size_t) s->n_faces * 4, &d.face_entity, ctx->stream)) != RT3_OK ||
        (rc = stage(spheres, s->spheres, (size_t) s->n_spheres * sizeof(rt3_sphere), &d.spheres, ctx->stream)) != RT3_OK ||
        (rc = stage(sphere_color, s->sphere_color, (size_t) s->n_spheres * 12, &d.sphere_color, ctx->stream)) != RT3_OK ||
        (rc = stage(sphere_material, s->sphere_material, (size_t) s->n_spheres * 4, &d.sphere_material, ctx->stream)) != RT3_OK ||
        (rc = stage(sphere_entity, s->sphere_entity, (size_t) s->n_spheres * 4, &d.sphere_entity, ctx->stream)) != RT3_OK ||
        (rc = stage(materials, s->materials, (size_t) s->n_materials * sizeof(rt3_material), &d.materials, ctx->stream)) != RT3_OK) {
        return rc;
    }
    RT3_CUDA(cudaEventRecord(ev.end, ctx->stream));
    rc = build_scene_on_device(ctx, d);
    if (rc != RT3_OK) { return rc; }
    float h2d = 0.f;
    RT3_CUDA(cudaEventElapsedTime(&h2d, ev.begin, ev.end));
    ctx->upload_h2d_ms = h2d;
    ctx->upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RT3_OK;
}

int rt3_scene_upload_device(rt3_ctx* ctx, const rt3_scene* s) {
    if (!ctx || !s) { return fail(RT3_ERR_INVALID, "ctx or scene is NULL"); }
    int rc = check_scene_args(s);
    if (rc != RT3_OK) { return rc; }
    if ((((uintptr_t) s->faces) | ((uintptr_t) s->vertices) | ((uintptr_t) s->spheres) | ((uintptr_t) s->materials)) & 15u) {
        return fail(RT3_ERR_INVALID, "device arrays of faces, vertices, spheres and materials must be 16-byte aligned");
    }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const auto t0 = std::chrono::steady_clock::now();
    rc = build_scene_on_device(ctx, *s);
    if (rc != RT3_OK) { return rc; }
    ctx->upload_h2d_ms = 0.0;
    ctx->upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RT3_OK;
}

int rt3_buffer_alloc(rt3_ctx* ctx, uint64_t bytes, void** device_ptr) {
    if (!ctx || !device_ptr) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    *device_ptr = nullptr;
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaMalloc(device_ptr, bytes ? (size_t) bytes : 1));
    return RT3_OK;
}

int rt3_buffer_free(rt3_ctx* ctx, void* device_ptr) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (!device_ptr) { return RT3_OK; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaStreamSynchronize(ctx->stream)); /* scene builds read these buffers on the context's stream */
    RT3_CUDA(cudaFree(device_ptr));
    return RT3_OK;
}

int rt3_buffer_write(rt3_ctx* ctx, void* device_dst, const void* host_src, uint64_t bytes) {
    if (!ctx || (bytes && (!device_dst || !host_src))) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    if (bytes) { RT3_CUDA(cudaMemcpyAsync(device_dst, host_src, (size_t) bytes, cudaMemcpyHostToDevice, ctx->stream)); }
    RT3_CUDA(cudaStreamSynchronize(ctx->stream)); /* the caller may reuse host_src */
    return RT3_OK;
}

int rt3_buffer_read(rt3_ctx* ctx, void* host_dst, const void* device_src, uint64_t bytes) {
    if (!ctx || (bytes && (!host_dst || !device_src))) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    if (bytes) { RT3_CUDA(cudaMemcpyAsync(host_dst, device_src, (size_t) bytes, cudaMemcpyDeviceToHost, ctx->stream)); }
    RT3_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT3_OK;
}

int rt3_render(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, uint32_t* host_frame) {
    return render_to_host(ctx, camera, params, host_frame, nullptr, nullptr, nullptr, false);
}

int rt3_render_aov(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, uint32_t* host_frame, uint32_t* host_hit_prim,
                   uint32_t* host_hit_entity, float* host_hit_t) {
    return render_to_host(ctx, camera, params, host_frame, host_hit_prim, host_hit_entity, host_hit_t, true);
}

int rt3_render_path_aovs(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, const rt3_path_aovs* out) {
    return render_path_aovs(ctx, camera, params, out);
}

int rt3_denoise(rt3_ctx* ctx, const rt3_denoise_params* params, uint32_t* host_frame, float* host_rgb) {
    return denoise(ctx, params, host_frame, host_rgb);
}

int rt3_denoise_temporal(rt3_ctx* ctx, const rt3_denoise_temporal_params* params, uint32_t* host_frame, float* host_rgb, float* host_history_length) {
    return denoise_temporal(ctx, params, host_frame, host_rgb, host_history_length);
}

uint64_t rt3_denoise_stage_words(uint32_t width, uint32_t height) {
    const uint64_t n = (uint64_t) width * height;
    if (n == 0) { return 0; }
    const uint64_t words = stage_fingerprint_offset(n) + 2ull * height;
    return words > 0xFFFFFFFFull ? 0 : words;
}

int rt3_denoise_stage(rt3_ctx* ctx, const rt3_denoise_params* params, uint64_t frame_tag, uint32_t* device_stage, void* cuda_stream) {
    return denoise_stage(ctx, params, frame_tag, device_stage, (cudaStream_t) cuda_stream);
}

int rt3_denoise_staged(rt3_ctx* ctx, const rt3_denoise_params* params, uint64_t frame_tag, const uint32_t* device_stage, uint32_t* host_frame,
                       float* host_rgb) {
    return denoise_staged(ctx, params, frame_tag, device_stage, host_frame, host_rgb);
}

int rt3_denoise_staged_temporal(rt3_ctx* ctx, const rt3_denoise_temporal_params* params, uint64_t frame_tag, const uint32_t* device_stage,
                                uint32_t* host_frame, float* host_rgb, float* host_history_length) {
    return denoise_staged_temporal(ctx, params, frame_tag, device_stage, host_frame, host_rgb, host_history_length);
}

int rt3_render_device(rt3_ctx* ctx, const rt3_camera* camera, const rt3_params* params, uint32_t* device_frame, void* cuda_stream) {
    rt3_kparams kp;
    int rc = check_render_args(ctx, camera, params, &kp);
    if (rc != RT3_OK) { return rc; }
    if (!device_frame) { return fail(RT3_ERR_INVALID, "device_frame is NULL"); }
    cudaStream_t stream = cuda_stream ? (cudaStream_t) cuda_stream : ctx->stream;
    return enqueue_render(ctx, camera, params, kp, device_frame, nullptr, nullptr, nullptr, stream);
}

uint32_t rt3_partition_rows(uint32_t height, uint32_t tile_rows, uint32_t part_index, uint32_t part_count) {
    return owned_rows(height, tile_rows, part_index, part_count);
}

static int partition_kparams(uint32_t width, uint32_t height, uint32_t tile_rows, uint32_t part_index, uint32_t part_count, rt3_kparams* kp) {
    rt3_params p;
    memset(&p, 0, sizeof p);
    p.width = width; p.height = height; p.mode = RT3_MODE_REFERENCE; p.tile_rows = tile_rows; p.part_index = part_index; p.part_count = part_count;
    return make_kparams(&p, kp);
}

int rt3_pack_partition(rt3_ctx* ctx, const uint32_t* device_frame, uint32_t* device_slab, uint32_t width, uint32_t height,
                       uint32_t tile_rows, uint32_t part_index, uint32_t part_count, void* cuda_stream) {
    if (!ctx || !device_frame || !device_slab) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    rt3_kparams kp;
    int rc = partition_kparams(width, height, tile_rows, part_index, part_count, &kp);
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    if (kp.n_pixels == 0) { return RT3_OK; }
    cudaStream_t stream = cuda_stream ? (cudaStream_t) cuda_stream : ctx->stream;
    pack_partition_kernel<<<(unsigned) ((kp.n_pixels + 255ull) / 256ull), 256, 0, stream>>>(kp, device_frame, device_slab);
    RT3_CUDA(cudaGetLastError());
    return RT3_OK;
}

int rt3_unpack_partition(rt3_ctx* ctx, const uint32_t* device_slab, uint32_t* device_frame, uint32_t width, uint32_t height,
                         uint32_t tile_rows, uint32_t part_index, uint32_t part_count, void* cuda_stream) {
    if (!ctx || !device_frame || !device_slab) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    rt3_kparams kp;
    int rc = partition_kparams(width, height, tile_rows, part_index, part_count, &kp);
    if (rc != RT3_OK) { return rc; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    if (kp.n_pixels == 0) { return RT3_OK; }
    cudaStream_t stream = cuda_stream ? (cudaStream_t) cuda_stream : ctx->stream;
    unpack_partition_kernel<<<(unsigned) ((kp.n_pixels + 255ull) / 256ull), 256, 0, stream>>>(kp, device_slab, device_frame);
    RT3_CUDA(cudaGetLastError());
    return RT3_OK;
}

int rt3_frame_alloc(rt3_ctx* ctx, uint64_t n_pixels, uint32_t** device_frame) {
    if (!ctx || !device_frame) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    *device_frame = nullptr;
    if (n_pixels == 0 || n_pixels > 0xFFFFFFFFull) { return fail(RT3_ERR_INVALID, "n_pixels must be in 1 .. 2^32-1"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    void* p = nullptr;
    /* a plain cudaMalloc: the IPC handle names the whole allocation, so the frame must be one */
    RT3_CUDA(cudaMalloc(&p, (size_t) n_pixels * sizeof(uint32_t)));
    cudaError_t e = cudaMemset(p, 0, (size_t) n_pixels * sizeof(uint32_t));
    if (e != cudaSuccess) { cudaFree(p); return fail(RT3_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e)); }
    *device_frame = (uint32_t*) p;
    return RT3_OK;
}

int rt3_frame_free(rt3_ctx* ctx, uint32_t* device_frame) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (!device_frame) { return RT3_OK; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaFree(device_frame));
    return RT3_OK;
}

int rt3_frame_export(rt3_ctx* ctx, const uint32_t* device_frame, unsigned char* handle_out) {
    if (!ctx || !device_frame || !handle_out) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    static_assert(sizeof(cudaIpcMemHandle_t) == RT3_IPC_HANDLE_BYTES, "RT3_IPC_HANDLE_BYTES must be the size of a CUDA IPC handle");
    RT3_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    RT3_CUDA(cudaIpcGetMemHandle(&h, const_cast<uint32_t*>(device_frame)));
    memcpy(handle_out, &h, sizeof h);
    return RT3_OK;
}

int rt3_frame_import(rt3_ctx* ctx, const unsigned char* handle, uint32_t** peer_frame) {
    if (!ctx || !handle || !peer_frame) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    *peer_frame = nullptr;
    RT3_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    void* p = nullptr;
    RT3_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *peer_frame = (uint32_t*) p;
    return RT3_OK;
}

int rt3_frame_release(rt3_ctx* ctx, uint32_t* peer_frame) {
    if (!ctx) { return fail(RT3_ERR_INVALID, "ctx is NULL"); }
    if (!peer_frame) { return RT3_OK; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaIpcCloseMemHandle(peer_frame));
    return RT3_OK;
}

int rt3_frame_attach(rt3_ctx* ctx, rt3_ctx* owner) {
    if (!ctx || !owner) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    if (ctx->device == owner->device) { return RT3_OK; }
    int can = 0;
    RT3_CUDA(cudaDeviceCanAccessPeer(&can, ctx->device, owner->device));
    if (!can) { return fail(RT3_ERR_CUDA, "device %d cannot access the memory of device %d", ctx->device, owner->device); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    cudaError_t e = cudaDeviceEnablePeerAccess(owner->device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { (void) cudaGetLastError(); e = cudaSuccess; }
    if (e != cudaSuccess) { (void) cudaGetLastError(); return fail(RT3_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d) failed: %s", owner->device, cudaGetErrorString(e)); }
    return RT3_OK;
}

int rt3_frame_read(rt3_ctx* ctx, const uint32_t* device_frame, uint32_t* host_frame, uint64_t n_pixels) {
    if (!ctx || !device_frame || !host_frame) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaMemcpyAsync(host_frame, device_frame, (size_t) n_pixels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    RT3_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT3_OK;
}

uint32_t rt3_uv_sphere_faces(uint32_t n_meridians, uint32_t n_parallels) { return n_parallels >= 3 ? uv_sphere_faces(n_meridians, n_parallels) : 0u; }
uint32_t rt3_uv_sphere_vertices(uint32_t n_meridians, uint32_t n_parallels) { return n_parallels >= 3 ? uv_sphere_vertices(n_meridians, n_parallels) : 0u; }

/* Counts and checks a batch of UV spheres. */
static int uv_batch_size(const rt3_uv_sphere* spheres, uint32_t n, unsigned long long* n_faces, unsigned long long* n_vertices) {
    *n_faces = 0; *n_vertices = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (spheres[i].n_parallels < 3 || spheres[i].n_meridians < 1) {
            return fail(RT3_ERR_INVALID, "sphere %u: needs n_parallels >= 3 and n_meridians >= 1 (got %u, %u)", i, spheres[i].n_parallels, spheres[i].n_meridians);
        }
        *n_faces += uv_sphere_faces(spheres[i].n_meridians, spheres[i].n_parallels);
        *n_vertices += uv_sphere_vertices(spheres[i].n_meridians, spheres[i].n_parallels);
    }
    return RT3_OK;
}

/* Sphere k's vertices go to d_vertices[vertex_slot + ...] and its faces to d_faces[face_slot + ...]; a face refers to
 * vertex j of its sphere as index_shift + (the vertex's position in d_vertices). Asynchronous on the context's stream. */
static int tessellate_on_device(rt3_ctx* ctx, const rt3_uv_sphere* spheres, uint32_t n, uint32_t vertex_slot, uint32_t face_slot, uint32_t index_shift,
                                uint4* d_faces, float4* d_vertices, uint32_t* d_entity) {
    uint32_t v0 = vertex_slot, f0 = face_slot;
    for (uint32_t i = 0; i < n; i++) {
        const rt3_uv_sphere& s = spheres[i];
        rt3_uv_sphere_dev d = { s.center[0], s.center[1], s.center[2], s.radius, s.n_meridians, s.n_parallels, s.color[0], s.color[1], s.color[2],
                                v0, f0, s.entity, index_shift };
        const uint32_t nv = uv_sphere_vertices(d.m, d.p), nf = uv_sphere_faces(d.m, d.p);
        uv_sphere_vertices_kernel<<<(nv + 255u) / 256u, 256, 0, ctx->stream>>>(d, d_vertices);
        RT3_CUDA(cudaGetLastError());
        uv_sphere_faces_kernel<<<(nf + 255u) / 256u, 256, 0, ctx->stream>>>(d, d_vertices, d_faces, d_entity);
        RT3_CUDA(cudaGetLastError());
        v0 += nv; f0 += nf;
    }
    return RT3_OK;
}

int rt3_tessellate_spheres(rt3_ctx* ctx, const rt3_uv_sphere* spheres, uint32_t n, uint32_t first_vertex, rt3_face* host_faces,
                           rt3_vertex* host_vertices, uint32_t* host_face_entity) {
    if (!ctx || (n && (!spheres || !host_faces || !host_vertices))) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    static_assert(sizeof(rt3_face) == 48 && sizeof(rt3_vertex) == 16, "flattened records must match the reference's GFace / glm::vec4");
    RT3_CUDA(cudaSetDevice(ctx->device));
    unsigned long long n_faces = 0, n_vertices = 0;
    int rc = uv_batch_size(spheres, n, &n_faces, &n_vertices);
    if (rc != RT3_OK) { return rc; }
    if (n_faces > 0x7FFFFFFFull || n_vertices + first_vertex > 0xFFFFFFFFull) { return fail(RT3_ERR_INVALID, "too many faces or vertices"); }
    if (n_faces == 0) { return RT3_OK; }
    DeviceBuffer<float4> d_vertices;
    DeviceBuffer<uint4> d_faces;
    DeviceBuffer<uint32_t> d_entity;
    if ((rc = d_vertices.reserve(n_vertices)) != RT3_OK || (rc = d_faces.reserve(3 * n_faces)) != RT3_OK || (rc = d_entity.reserve(n_faces)) != RT3_OK) { return rc; }
    if ((rc = tessellate_on_device(ctx, spheres, n, 0u, 0u, first_vertex, d_faces.ptr, d_vertices.ptr, d_entity.ptr)) != RT3_OK) { return rc; }
    RT3_CUDA(cudaMemcpyAsync(host_vertices, d_vertices.ptr, n_vertices * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    RT3_CUDA(cudaMemcpyAsync(host_faces, d_faces.ptr, n_faces * 48, cudaMemcpyDeviceToHost, ctx->stream));
    if (host_face_entity) { RT3_CUDA(cudaMemcpyAsync(host_face_entity, d_entity.ptr, n_faces * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream)); }
    RT3_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT3_OK;
}

int rt3_tessellate_spheres_device(rt3_ctx* ctx, const rt3_uv_sphere* spheres, uint32_t n, uint32_t first_vertex, uint32_t first_face,
                                  rt3_face* device_faces, rt3_vertex* device_vertices, uint32_t* device_face_entity) {
    if (!ctx || (n && (!spheres || !device_faces || !device_vertices))) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    if ((((uintptr_t) device_faces) | ((uintptr_t) device_vertices)) & 15u) { return fail(RT3_ERR_INVALID, "device arrays must be 16-byte aligned"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    unsigned long long n_faces = 0, n_vertices = 0;
    int rc = uv_batch_size(spheres, n, &n_faces, &n_vertices);
    if (rc != RT3_OK) { return rc; }
    if (n_faces + first_face > 0x7FFFFFFFull || n_vertices + first_vertex > 0xFFFFFFFFull) { return fail(RT3_ERR_INVALID, "too many faces or vertices"); }
    return tessellate_on_device(ctx, spheres, n, first_vertex, first_face, 0u, reinterpret_cast<uint4*>(device_faces), reinterpret_cast<float4*>(device_vertices),
                                device_face_entity);
}

int rt3_frame_bytes(rt3_ctx* ctx, const uint32_t* device_frame, unsigned char* device_out, uint32_t width, uint32_t height, uint32_t channels,
                    void* cuda_stream) {
    if (!ctx || !device_frame || !device_out) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    if (channels != 3 && channels != 4) { return fail(RT3_ERR_INVALID, "channels must be 3 (RGB) or 4 (RGBA), got %u", channels); }
    if (((uintptr_t) device_frame & 15u) || ((uintptr_t) device_out & 15u)) { return fail(RT3_ERR_INVALID, "device buffers must be 16-byte aligned"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const unsigned long long n = (unsigned long long) width * height;
    if (n == 0) { return RT3_OK; }
    cudaStream_t stream = cuda_stream ? (cudaStream_t) cuda_stream : ctx->stream;
    const unsigned grid = (unsigned) (((n + 3ull) / 4ull + 255ull) / 256ull);
    if (channels == 4) { frame_bytes_kernel<4><<<grid, 256, 0, stream>>>(device_frame, device_out, n); }
    else { frame_bytes_kernel<3><<<grid, 256, 0, stream>>>(device_frame, device_out, n); }
    RT3_CUDA(cudaGetLastError());
    return RT3_OK;
}

int rt3_read_radiance(rt3_ctx* ctx, float* host_rgb, uint32_t width, uint32_t height) {
    if (!ctx || !host_rgb) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    if (!ctx->accum_valid) { return fail(RT3_ERR_INVALID, "no path-traced render on this context to read the radiance of"); }
    const rt3_kparams& kp = ctx->accum_kp;
    if (kp.width != width || kp.height != height) {
        return fail(RT3_ERR_INVALID, "the last path-traced frame was %ux%u, not %ux%u", kp.width, kp.height, width, height);
    }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t) kp.width * kp.height * 3;
    DeviceBuffer<float> rgb;
    int rc = rgb.reserve(n);
    if (rc != RT3_OK) { return rc; }
    cudaStream_t stream = accum_stream(ctx);
    RT3_CUDA(cudaMemsetAsync(rgb.ptr, 0, n * sizeof(float), stream));
    if (kp.n_pixels) {
        radiance_kernel<<<(unsigned) ((kp.n_pixels + 255ull) / 256ull), 256, 0, stream>>>(kp, ctx->accum.ptr, rgb.ptr);
        RT3_CUDA(cudaGetLastError());
    }
    RT3_CUDA(cudaMemcpyAsync(host_rgb, rgb.ptr, n * sizeof(float), cudaMemcpyDeviceToHost, stream));
    RT3_CUDA(cudaStreamSynchronize(stream));
    return RT3_OK;
}

int rt3_get_stats(rt3_ctx* ctx, rt3_stats* out) {
    if (!ctx || !out) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    int rc = collect_stats(ctx);
    if (rc != RT3_OK) { return rc; }
    *out = ctx->stats;
    /* the scene build is not part of a render: reported from the most recent upload on this context */
    out->h2d_ms = ctx->upload_h2d_ms;
    out->upload_ms = ctx->upload_ms;
    out->upload_device_ms = ctx->upload_device_ms;
    return RT3_OK;
}

#ifdef RT3_SURVIVOR_STATS
/* Debug build only: reads and clears the level-1 survivor statistics (rt3_kernels.cuh g_survivor_stats). */
int rt3_debug_survivor_stats(rt3_ctx* ctx, unsigned long long* out4) {
    if (!ctx || !out4) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    RT3_CUDA(cudaSetDevice(ctx->device));
    RT3_CUDA(cudaDeviceSynchronize());
    RT3_CUDA(cudaMemcpyFromSymbol(out4, g_survivor_stats, 4 * sizeof(unsigned long long)));
    const unsigned long long zero[4] = { 0, 0, 0, 0 };
    RT3_CUDA(cudaMemcpyToSymbol(g_survivor_stats, zero, sizeof zero));
    return RT3_OK;
}
#endif

int rt3_measure_fma_peak(rt3_ctx* ctx, double* tflops_out) {
    if (!ctx || !tflops_out) { return fail(RT3_ERR_INVALID, "NULL argument"); }
    int rc0 = collect_stats(ctx);
    if (rc0 != RT3_OK) { return rc0; }
    RT3_CUDA(cudaSetDevice(ctx->device));
    const int threads = 256, blocks = ctx->sm_count * 8, iters = 1 << 15;
    DeviceBuffer<float> out;
    int rc = out.reserve((size_t) threads * blocks);
    if (rc != RT3_OK) { return rc; }
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        RT3_CUDA(cudaEventRecord(ctx->ev_begin, ctx->stream));
        fma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(out.ptr, 0.999f, 0.001f, iters);
        RT3_CUDA(cudaGetLastError());
        RT3_CUDA(cudaEventRecord(ctx->ev_end, ctx->stream));
        RT3_CUDA(cudaStreamSynchronize(ctx->stream));
        float ms = 0.f;
        RT3_CUDA(cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
        double flops = 2.0 * 16.0 * (double) iters * threads * blocks;
        double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) { best = tf; }
    }
    *tflops_out = best;
    return RT3_OK;
}

}  // extern "C"
