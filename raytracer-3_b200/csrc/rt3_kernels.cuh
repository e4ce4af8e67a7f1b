/* rt3_kernels.cuh — the sm_100a kernels of the render core.
 *
 *   reference_kernel   : the reference's ray caster (one un-jittered primary
 *                        ray per pixel, closest hit, flat colour / sky, AOVs).
 *   pathtrace_kernel   : persistent multi-bounce path tracer with in-warp path
 *                        regeneration and fixed-point accumulation.
 *   resolve_kernel     : mean over samples, gamma, 8-bit pack.
 *   radiance_kernel    : the same mean as linear float RGB (AOV dump).
 *   pack/unpack kernels: frame <-> partition slab for the frame-end gather.
 *   fma_peak_kernel    : FFMA throughput probe (roofline denominator).
 *
 * Both render kernels run the same sweep (rt3_device.cuh): per primitive pair
 * and ray three packed FMAs of a conservative slab test, the records coming
 * from the constant bank through uniform registers (scenes up to
 * RT3_CONST_PRIMS) or from TMA-streamed shared-memory tiles; the exact tests
 * run only on the survivors. With RT3_FLAG_BVH (template parameter ACCEL) the
 * sweep is replaced by the hierarchy traversal of rt3_bvh.cuh, same results.
 */
#pragma once

#include "rt3_device.cuh"
#include "rt3_bvh.cuh"

struct rt3_kparams {
    uint32_t width, height;
    uint32_t spp, max_depth, seed, flags;
    uint32_t first_sample;        /* this launch renders samples [first_sample, first_sample + spp) of every pixel */
    uint32_t resolve_spp;         /* samples behind the accumulators when the frame is resolved */
    uint32_t tile_rows, part_index, part_count;
    uint32_t owned_rows;          /* rows this partition renders */
    unsigned long long n_pixels;  /* owned_rows * width */
    unsigned long long n_items;   /* n_pixels * spp */
    uint32_t resident;            /* 1: the whole prefilter array is kept in shared memory */
};

/* Compact owned-row index -> global row (row tiles dealt round-robin to partitions). */
__device__ __forceinline__ uint32_t owned_row_to_global(const rt3_kparams& P, uint32_t local_row) {
    uint32_t lt = local_row / P.tile_rows, within = local_row - lt * P.tile_rows;
    return (lt * P.part_count + P.part_index) * P.tile_rows + within;
}

/* Shared-memory layout.
 *   resident (constant-bank) scenes: [survivor masks] [path slots]
 *   streamed scenes:                 [mbarriers (64 B)] [2 stages x (pair_xy tile, pair_w tile)] [survivor masks] [path slots]
 * The path slots (path tracer only) hold the state of every ray of every thread, one 32-bit word per
 * field, laid out [slot][field][thread] so that a warp's accesses to a field are conflict-free. */
struct rt3_smem_view {
    uint64_t* bars;   /* streamed: one "tile landed" mbarrier per stage */
    float4* tile_xy;  /* streamed: 2 stages of RT3_TILE_PRIMS / 2 pair records */
    float2* tile_w;
    uint32_t* masks;  /* RT3_RAYS * RT3_CHUNK_WORDS * RT3_CTA_THREADS words */
    uint32_t* slots;  /* RT3_RAYS * RT3_SLOT_FIELDS * RT3_CTA_THREADS words */
};

enum { RT3_F_OX, RT3_F_OY, RT3_F_OZ, RT3_F_DX, RT3_F_DY, RT3_F_DZ, RT3_F_TX, RT3_F_TY, RT3_F_TZ, RT3_F_KEY, RT3_F_PIX,
       RT3_F_BOUNCE /* RT3_NO_HIT: the slot is free */, RT3_F_BEST_T, RT3_F_BEST_PRIM, RT3_SLOT_FIELDS };
#define RT3_SLOT_BYTES (RT3_RAYS * RT3_SLOT_FIELDS * RT3_CTA_THREADS * 4)

#define RT3_TILE_PAIRS (RT3_TILE_PRIMS / 2)
#define RT3_TILE_XY_BYTES (RT3_TILE_PAIRS * 16)
#define RT3_TILE_W_BYTES (RT3_TILE_PAIRS * 8)

/* path_slots: the path tracer (RT3_RAYS rays per thread + their slots); otherwise the reference-mode kernel (RT3_REF_RAYS rays per thread). */
__host__ __device__ inline size_t rt3_smem_bytes(bool resident, bool path_slots) {
    const size_t masks = path_slots ? (size_t) RT3_MASK_BYTES : (size_t) RT3_MASK_BYTES_FOR(RT3_REF_RAYS);
    return (resident ? masks : (size_t) 64 + 2 * (RT3_TILE_XY_BYTES + RT3_TILE_W_BYTES) + masks) + (path_slots ? (size_t) RT3_SLOT_BYTES : 0);
}

/* Hierarchy kernels keep no survivor masks: their shared memory is the path slots alone, which
 * leaves the rest of the SM's 256 KB to the L1 the node records are read through. */
__host__ __device__ inline size_t rt3_accel_smem_bytes(bool path_slots) { return path_slots ? (size_t) RT3_SLOT_BYTES : 0; }
/* ... plus, for the binned traversal, the sort scratch (rt3_bin_scratch, defined with the traversal below): one KB */
#define RT3_BIN_SCRATCH_BYTES 1024

template <bool RESIDENT, bool ACCEL = false, int MASK_BYTES = RT3_MASK_BYTES>
__device__ __forceinline__ rt3_smem_view smem_view(unsigned char* base) {
    rt3_smem_view v;
    if (ACCEL) {
        v.bars = nullptr; v.tile_xy = nullptr; v.tile_w = nullptr; v.masks = nullptr;
        v.slots = reinterpret_cast<uint32_t*>(base);
    } else if (RESIDENT) {
        v.bars = nullptr; v.tile_xy = nullptr; v.tile_w = nullptr;
        v.masks = reinterpret_cast<uint32_t*>(base);
        v.slots = reinterpret_cast<uint32_t*>(base + MASK_BYTES);
    } else {
        v.bars = reinterpret_cast<uint64_t*>(base);
        v.tile_xy = reinterpret_cast<float4*>(base + 64);
        v.tile_w = reinterpret_cast<float2*>(base + 64 + 2 * RT3_TILE_XY_BYTES);
        v.masks = reinterpret_cast<uint32_t*>(base + 64 + 2 * (RT3_TILE_XY_BYTES + RT3_TILE_W_BYTES));
        v.slots = reinterpret_cast<uint32_t*>(base + 64 + 2 * (RT3_TILE_XY_BYTES + RT3_TILE_W_BYTES) + MASK_BYTES);
    }
    return v;
}

/* Arms the streaming barriers (streamed scenes only). */
template <bool RESIDENT>
__device__ __forceinline__ void scene_prologue(const rt3_smem_view& sm) {
    if (RESIDENT) { return; }
    if (threadIdx.x == 0) {
        mbar_init(&sm.bars[0], 1);
        mbar_init(&sm.bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
}

/* Streamed scenes: one thread starts the bulk asynchronous copies (TMA, SASS UBLKCP) of tile `t` into `stage`. */
__device__ __forceinline__ void fetch_tile(const rt3_scene_view& S, const rt3_smem_view& sm, uint32_t t, uint32_t stage) {
    const uint32_t first_pair = t * RT3_TILE_PAIRS, total_pairs = S.n_prims_padded / 2;
    const uint32_t n = total_pairs - first_pair < RT3_TILE_PAIRS ? total_pairs - first_pair : RT3_TILE_PAIRS;
    mbar_expect_tx(&sm.bars[stage], n * 24u);
    bulk_copy_g2s(sm.tile_xy + (size_t) stage * RT3_TILE_PAIRS, S.pair_xy + first_pair, n * 16u, &sm.bars[stage]);
    bulk_copy_g2s(sm.tile_w + (size_t) stage * RT3_TILE_PAIRS, S.pair_w + first_pair, n * 8u, &sm.bars[stage]);
}

/* Closest hit of the thread's rays against the whole scene. For streamed
 * scenes every thread of the CTA must call this together (tile barriers);
 * `phase` carries the mbarrier parities across calls. */
template <bool PATH_MODE, bool RESIDENT, bool SPHERES_ONLY, int R>
__device__ __forceinline__ void sweep_scene(const rt3_scene_view& S, const rt3_smem_view& sm, uint32_t& phase,
                                            const rt3_vec3 (&o)[R], const rt3_vec3 (&d)[R], const rt3_vec3 (&dn)[R],
                                            const bool (&live)[R], rt3_hit (&best)[R]) {
    rt3_ray_filter f[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        f[r] = make_ray_filter(S, o[r], dn[r]);
        best[r].t = __int_as_float(0x7f800000);
        best[r].prim = RT3_NO_HIT;
    }
    if (RESIDENT) {
        sweep_range<PATH_MODE, true, SPHERES_ONLY, R>(S, nullptr, nullptr, 0u, 0u, S.n_prims_padded, f, o, d, live, sm.masks, best);
        return;
    }
    const uint32_t n_tiles = (S.n_prims_padded + RT3_TILE_PRIMS - 1) / RT3_TILE_PRIMS;
    if (threadIdx.x == 0 && n_tiles > 0) { fetch_tile(S, sm, 0u, 0u); }
    for (uint32_t t = 0; t < n_tiles; t++) {
        const uint32_t stage = t & 1u;
        /* stage^1 was last read for tile t-1; the __syncthreads below ordered those reads before this copy */
        if (threadIdx.x == 0 && t + 1 < n_tiles) { fetch_tile(S, sm, t + 1, stage ^ 1u); }
        mbar_wait(&sm.bars[stage], (phase >> stage) & 1u);
        phase ^= 1u << stage;
        const uint32_t first = t * RT3_TILE_PRIMS;
        const uint32_t n = S.n_prims_padded - first < RT3_TILE_PRIMS ? S.n_prims_padded - first : RT3_TILE_PRIMS;
        sweep_range<PATH_MODE, false, SPHERES_ONLY, R>(S, sm.tile_xy + (size_t) stage * RT3_TILE_PAIRS, sm.tile_w + (size_t) stage * RT3_TILE_PAIRS, 0u, first, n,
                                      f, o, d, live, sm.masks, best);
        __syncthreads();
    }
}

/* ---- path slots in shared memory ------------------------------------------ */

__device__ __forceinline__ uint32_t& slot_word(const rt3_smem_view& sm, int r, int field) {
    return sm.slots[(r * RT3_SLOT_FIELDS + field) * RT3_CTA_THREADS + threadIdx.x];
}
__device__ __forceinline__ float slot_float(const rt3_smem_view& sm, int r, int field) { return __uint_as_float(slot_word(sm, r, field)); }
__device__ __forceinline__ rt3_vec3 slot_vec(const rt3_smem_view& sm, int r, int field) {
    return v3(slot_float(sm, r, field), slot_float(sm, r, field + 1), slot_float(sm, r, field + 2));
}
__device__ __forceinline__ void slot_store_vec(const rt3_smem_view& sm, int r, int field, rt3_vec3 v) {
    slot_word(sm, r, field) = __float_as_uint(v.x); slot_word(sm, r, field + 1) = __float_as_uint(v.y); slot_word(sm, r, field + 2) = __float_as_uint(v.z);
}

/* Level-1 constants of every slot's ray; a free slot gets a filter nothing survives (a = +inf). */
__device__ __forceinline__ void slot_filters(const rt3_scene_view& S, const rt3_smem_view& sm, rt3_ray_filter (&f)[RT3_RAYS]) {
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) {
        f[r] = make_ray_filter(S, slot_vec(sm, r, RT3_F_OX), slot_vec(sm, r, RT3_F_DX));
        if (slot_word(sm, r, RT3_F_BOUNCE) == RT3_NO_HIT) { f[r].u1 = 0.0f; f[r].u2 = 0.0f; f[r].nou = __int_as_float(0x7f800000); }
    }
}

#ifdef RT3_SURVIVOR_STATS
/* Debug build only (profiles/survivors.py): how many primitives level 1 lets through. [0] survivors (ray, primitive) pairs,
 * [1] sum over warp-drains of the largest per-lane survivor count (= iterations the warp spends in the drain loop),
 * [2] warp-drains, [3] lanes with a live ray in them. */
__device__ unsigned long long g_survivor_stats[4];
__device__ __forceinline__ void count_survivors(const uint32_t* __restrict__ masks, uint32_t n_words, uint32_t nz, bool live) {
    uint32_t mine = 0;
    for (uint32_t wd = 0; wd < n_words; wd++) { if ((nz >> (n_words - 1u - wd)) & 1u) { mine += (uint32_t) __popc(masks[wd * RT3_CTA_THREADS]); } }
    const uint32_t total = __reduce_add_sync(0xffffffffu, mine), most = __reduce_max_sync(0xffffffffu, mine);
    const uint32_t lanes = (uint32_t) __popc(__ballot_sync(0xffffffffu, live));
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&g_survivor_stats[0], (unsigned long long) total); atomicAdd(&g_survivor_stats[1], (unsigned long long) most);
        atomicAdd(&g_survivor_stats[2], 1ull); atomicAdd(&g_survivor_stats[3], (unsigned long long) lanes);
    }
}
#endif

/* Drains one chunk for every slot, one slot at a time from a single copy of the code. */
template <bool SPHERES_ONLY>
__device__ __forceinline__ void drain_slots(const rt3_scene_view& S, const rt3_smem_view& sm, uint32_t first_prim, uint32_t n_pairs,
                                            const rt3_ray_filter (&f)[RT3_RAYS], const uint32_t (&nz)[RT3_RAYS]) {
    const uint32_t n_words = (n_pairs + RT3_WORD_PRIMS / 2 - 1) / (RT3_WORD_PRIMS / 2);
    static_assert(RT3_RAYS * RT3_CHUNK_WORDS <= 64, "survivor summaries are packed into 64 bits");
    unsigned long long packed = 0ull;
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) { packed |= (unsigned long long) nz[r] << (r * RT3_CHUNK_WORDS); }
#pragma unroll 1
    for (int r = 0; r < RT3_RAYS; r++) {
        const uint32_t mine = (uint32_t) (packed >> (r * RT3_CHUNK_WORDS)) & ((1u << RT3_CHUNK_WORDS) - 1u);
        rt3_hit best;
        best.t = slot_float(sm, r, RT3_F_BEST_T); best.prim = slot_word(sm, r, RT3_F_BEST_PRIM);
        rt3_ray_filter fr = f[0]; /* level 2 is only needed for faces; rebuilt below for the slot at hand */
        const rt3_vec3 o = slot_vec(sm, r, RT3_F_OX), d = slot_vec(sm, r, RT3_F_DX);
        if (!SPHERES_ONLY) { fr = make_ray_filter(S, o, d); }
#ifdef RT3_SURVIVOR_STATS
        count_survivors(sm.masks + r * RT3_CHUNK_WORDS * RT3_CTA_THREADS + threadIdx.x, n_words, mine, slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT);
#endif
        drain_chunk<true, SPHERES_ONLY>(S, first_prim, n_words, fr, o, d, sm.masks + r * RT3_CHUNK_WORDS * RT3_CTA_THREADS + threadIdx.x, mine, best);
        slot_word(sm, r, RT3_F_BEST_T) = __float_as_uint(best.t); slot_word(sm, r, RT3_F_BEST_PRIM) = best.prim;
    }
}

/* Closest hit of every slot's ray against the whole scene (results in the slots' BEST fields). */
template <bool RESIDENT, bool SPHERES_ONLY>
__device__ __forceinline__ void sweep_slots(const rt3_scene_view& S, const rt3_smem_view& sm, uint32_t& phase) {
    constexpr uint32_t CHUNK_PAIRS = RT3_CHUNK_WORDS * RT3_WORD_PRIMS / 2;
    rt3_ray_filter f[RT3_RAYS];
    slot_filters(S, sm, f);
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) { slot_word(sm, r, RT3_F_BEST_T) = 0x7f800000u; slot_word(sm, r, RT3_F_BEST_PRIM) = RT3_NO_HIT; }
    if (RESIDENT) {
        const uint32_t n_pairs = S.n_prims_padded / 2;
        for (uint32_t p0 = 0; p0 < n_pairs; p0 += CHUNK_PAIRS) {
            uint32_t nz[RT3_RAYS];
            const uint32_t np = n_pairs - p0 < CHUNK_PAIRS ? n_pairs - p0 : CHUNK_PAIRS;
            sweep_chunk<true, RT3_RAYS>(nullptr, nullptr, p0, np, f, sm.masks, nz);
            drain_slots<SPHERES_ONLY>(S, sm, 2u * p0, np, f, nz);
        }
        return;
    }
    const uint32_t n_tiles = (S.n_prims_padded + RT3_TILE_PRIMS - 1) / RT3_TILE_PRIMS;
    if (threadIdx.x == 0 && n_tiles > 0) { fetch_tile(S, sm, 0u, 0u); }
    for (uint32_t t = 0; t < n_tiles; t++) {
        const uint32_t stage = t & 1u;
        if (threadIdx.x == 0 && t + 1 < n_tiles) { fetch_tile(S, sm, t + 1, stage ^ 1u); }
        mbar_wait(&sm.bars[stage], (phase >> stage) & 1u);
        phase ^= 1u << stage;
        const uint32_t first = t * RT3_TILE_PRIMS;
        const uint32_t n_pairs = (S.n_prims_padded - first < RT3_TILE_PRIMS ? S.n_prims_padded - first : RT3_TILE_PRIMS) / 2;
        const float4* xy = sm.tile_xy + (size_t) stage * RT3_TILE_PAIRS;
        const float2* w = sm.tile_w + (size_t) stage * RT3_TILE_PAIRS;
        for (uint32_t p0 = 0; p0 < n_pairs; p0 += CHUNK_PAIRS) {
            uint32_t nz[RT3_RAYS];
            const uint32_t np = n_pairs - p0 < CHUNK_PAIRS ? n_pairs - p0 : CHUNK_PAIRS;
            sweep_chunk<false, RT3_RAYS>(xy, w, p0, np, f, sm.masks, nz);
            drain_slots<SPHERES_ONLY>(S, sm, first + 2u * p0, np, f, nz);
        }
        __syncthreads();
    }
}

/* Any slot of the CTA, not just the calling thread's: */
__device__ __forceinline__ uint32_t& slot_word_at(const rt3_smem_view& sm, uint32_t r, int field, uint32_t t) {
    return sm.slots[(r * RT3_SLOT_FIELDS + field) * RT3_CTA_THREADS + t];
}
__device__ __forceinline__ rt3_vec3 slot_vec_at(const rt3_smem_view& sm, uint32_t r, int field, uint32_t t) {
    return v3(__uint_as_float(slot_word_at(sm, r, field, t)), __uint_as_float(slot_word_at(sm, r, field + 1, t)), __uint_as_float(slot_word_at(sm, r, field + 2, t)));
}

/* The tail of a frame. When the item counter has run dry a warp keeps sweeping for its last few paths, and a sweep costs the same
 * whether 64 or 3 of its slots hold a ray (level 1 alone is 1 600 warp instructions per slot pair): the last generation of paths
 * of a frame has members 25-30 segments long, so every frame ends with ~0.5 ms of nearly empty sweeps -- 0.4 % of a one-GPU
 * frame, 3 % of an eighth of it. With at most RT3_TAIL_RAYS rays left, the warp turns the loop inside out: one ray at a time, the
 * 32 lanes share the PRIMITIVES (lane l tests l, l + 32, ... with the exact tests, no prefilter) and a shuffle reduction picks the
 * closest hit, ties to the lower id like everywhere else. Same exact tests, same rule: same result bit for bit. */
#ifndef RT3_TAIL_RAYS
#define RT3_TAIL_RAYS 8
#endif
/* Slots of this warp that hold a ray (the same number in every lane). */
__device__ __forceinline__ uint32_t warp_live_slots(const rt3_smem_view& sm) {
    uint32_t n = 0;
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) { n += (uint32_t) __popc(__ballot_sync(0xffffffffu, slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT)); }
    return n;
}

__device__ __noinline__ void sweep_slots_by_primitive(const rt3_scene_view& S, const rt3_smem_view& sm) {
    const uint32_t lane = threadIdx.x & 31u, column0 = threadIdx.x & ~31u;
#pragma unroll 1
    for (uint32_t r = 0; r < RT3_RAYS; r++) {
        uint32_t todo = __ballot_sync(0xffffffffu, slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT);
        while (todo) {
            const uint32_t t = column0 + (uint32_t) __ffs((int) todo) - 1u; /* the owner's column: every lane reads the same words (broadcast) */
            todo &= todo - 1u;
            const rt3_vec3 o = slot_vec_at(sm, r, RT3_F_OX, t), d = slot_vec_at(sm, r, RT3_F_DX, t);
            rt3_hit best;
            best.t = __int_as_float(0x7f800000); best.prim = RT3_NO_HIT;
            for (uint32_t prim = lane; prim < S.n_prims; prim += 32u) {
                if (prim < S.n_faces) { exact_face<false>(S, prim, o, d, RT3_TMIN, best); }
                else { exact_sphere_path<false>(prim, __ldg(&S.spheres[prim - S.n_faces]), o, d, best); }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                rt3_hit other;
                other.t = __shfl_xor_sync(0xffffffffu, best.t, off); other.prim = __shfl_xor_sync(0xffffffffu, best.prim, off);
                if (other.prim != RT3_NO_HIT && closer<false>(other.t, other.prim, best)) { best = other; }
            }
            if (lane == 0) { slot_word_at(sm, r, RT3_F_BEST_T, t) = __float_as_uint(best.t); slot_word_at(sm, r, RT3_F_BEST_PRIM, t) = best.prim; }
        }
    }
    __syncwarp();
}

/* Hierarchy traversal for every live slot (results in the slots' BEST fields). */
__device__ __forceinline__ void traverse_slots(const rt3_scene_view& S, const rt3_bvh_view& B, const rt3_smem_view& sm, uint32_t& visits, uint32_t& tests) {
#pragma unroll 1
    for (int r = 0; r < RT3_RAYS; r++) {
        if (slot_word(sm, r, RT3_F_BOUNCE) == RT3_NO_HIT) { continue; }
        rt3_hit best;
        bvh_closest_hit<true>(S, B, slot_vec(sm, r, RT3_F_OX), slot_vec(sm, r, RT3_F_DX), best, visits, tests);
        slot_word(sm, r, RT3_F_BEST_T) = __float_as_uint(best.t); slot_word(sm, r, RT3_F_BEST_PRIM) = best.prim;
    }
}

/* ---- binned traversal (hierarchy kernels of scenes with a face tree) --------------------------------------------
 * The average ray of a mesh-in-a-landscape scene (BASELINE C3) is cheap -- it misses the mesh's box and is done after
 * two or three node visits -- while a ray that enters the mesh walks forty nodes; with every lane walking its own
 * slot's ray, the few expensive rays of a warp keep it busy with a handful of lanes active (9 of 32 measured in
 * round 1). Here the CTA sorts its 256 in-flight rays by that one bit before each traversal: the rays that enter the
 * face tree's root box first, then the others; warps then take 32 consecutive rays of that order at a time
 * ("passes", handed out by a shared counter), so the expensive rays travel together in few, full warps and the
 * cheap ones in warps that finish at once. The bit is a scheduling hint only: results do not depend on it.
 *
 * Scratch shared memory behind the path slots: */
struct rt3_bin_scratch {
    float root_lo[3], root_hi[3];     /* box of the face tree's root (union of its two child boxes) */
    uint32_t counts[RT3_CTA_THREADS / 32][4]; /* per warp: expensive rays in slot 0, slot 1; cheap rays in slot 0, slot 1 */
    uint32_t next_pass;
    uint32_t pad;
    uint16_t order[RT3_RAYS * RT3_CTA_THREADS]; /* ray ids (slot * RT3_CTA_THREADS + thread), expensive first */
};
static_assert(sizeof(rt3_bin_scratch) <= RT3_BIN_SCRATCH_BYTES, "the sort scratch must fit its reservation");


/* Does the ray meet the box at all (t >= 0)? Plain slab test; NaNs (a direction component of 0 on a slab plane) count as a hit. */
__device__ __forceinline__ bool ray_meets_box(rt3_vec3 o, rt3_vec3 d, const float* lo, const float* hi) {
    const float ix = 1.0f / d.x, iy = 1.0f / d.y, iz = 1.0f / d.z;
    const float x0 = (lo[0] - o.x) * ix, x1 = (hi[0] - o.x) * ix, y0 = (lo[1] - o.y) * iy, y1 = (hi[1] - o.y) * iy, z0 = (lo[2] - o.z) * iz, z1 = (hi[2] - o.z) * iz;
    const float tin = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
    const float tout = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
    return !(tin > tout * 1.0001f) && !(tout < 0.0f);
}

/* Thread 0 of the CTA, once per kernel. */
__device__ __forceinline__ void bin_prologue(const rt3_bvh_view& B, rt3_bin_scratch* bin) {
    if (threadIdx.x == 0) {
        const int32_t root = B.tree[0].root;
        const float4 n0 = __ldg(&B.nodes[4 * root + 0]), n1 = __ldg(&B.nodes[4 * root + 1]), n2 = __ldg(&B.nodes[4 * root + 2]);
        /* fminf / fmaxf ignore the NaN boxes of primitives that can never be hit */
        bin->root_lo[0] = fminf(n0.x, n1.z); bin->root_lo[1] = fminf(n0.y, n1.w); bin->root_lo[2] = fminf(n0.z, n2.x);
        bin->root_hi[0] = fmaxf(n0.w, n2.y); bin->root_hi[1] = fmaxf(n1.x, n2.z); bin->root_hi[2] = fmaxf(n1.y, n2.w);
        bin->next_pass = 0u;
    }
    __syncthreads();
}

/* One traversal step of the whole CTA: sort the in-flight rays, traverse them pass by pass, leave every closest hit in its
 * slot. Returns false (for every thread of the CTA alike) when no slot of the CTA holds a ray any more. */
__device__ __forceinline__ bool traverse_slots_binned(const rt3_scene_view& S, const rt3_bvh_view& B, const rt3_smem_view& sm, rt3_bin_scratch* bin,
                                                      uint32_t& visits, uint32_t& tests) {
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, lane_lt = (1u << lane) - 1u;
    constexpr uint32_t WARPS = RT3_CTA_THREADS / 32;
    static_assert(RT3_RAYS == 2, "the binned traversal is written for two slots per thread");
    uint32_t heavy[RT3_RAYS], light[RT3_RAYS];
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) {
        const bool live = slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT;
        const bool meets = live && ray_meets_box(slot_vec(sm, r, RT3_F_OX), slot_vec(sm, r, RT3_F_DX), bin->root_lo, bin->root_hi);
        heavy[r] = __ballot_sync(0xffffffffu, meets);
        light[r] = __ballot_sync(0xffffffffu, live && !meets);
    }
    if (lane == 0) {
        bin->counts[warp][0] = (uint32_t) __popc(heavy[0]); bin->counts[warp][1] = (uint32_t) __popc(heavy[1]);
        bin->counts[warp][2] = (uint32_t) __popc(light[0]); bin->counts[warp][3] = (uint32_t) __popc(light[1]);
    }
    __syncthreads();
    uint32_t n_heavy = 0, n_light = 0, heavy_before = 0, light_before = 0;
#pragma unroll
    for (uint32_t w = 0; w < WARPS; w++) {
        const uint32_t h = bin->counts[w][0] + bin->counts[w][1], l = bin->counts[w][2] + bin->counts[w][3];
        if (w < warp) { heavy_before += h; light_before += l; }
        n_heavy += h; n_light += l;
    }
    const uint32_t n_live = n_heavy + n_light;
    if (n_live == 0u) { return false; }
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) {
        const uint32_t id = (uint32_t) r * RT3_CTA_THREADS + threadIdx.x;
        const uint32_t at_heavy = heavy_before + (r ? (uint32_t) __popc(heavy[0]) : 0u) + (uint32_t) __popc(heavy[r] & lane_lt);
        const uint32_t at_light = n_heavy + light_before + (r ? (uint32_t) __popc(light[0]) : 0u) + (uint32_t) __popc(light[r] & lane_lt);
        RT3_ASSERT(!((heavy[r] >> lane) & 1u) || at_heavy < n_heavy);
        RT3_ASSERT(!((light[r] >> lane) & 1u) || (at_light >= n_heavy && at_light < n_live));
        if ((heavy[r] >> lane) & 1u) { bin->order[at_heavy] = (uint16_t) id; }
        if ((light[r] >> lane) & 1u) { bin->order[at_light] = (uint16_t) id; }
    }
    __syncthreads();
    for (;;) {
        uint32_t pass = 0;
        if (lane == 0) { pass = atomicAdd(&bin->next_pass, 1u); }
        pass = __shfl_sync(0xffffffffu, pass, 0);
        if (pass * 32u >= n_live) { break; }
        const uint32_t idx = pass * 32u + lane;
        if (idx < n_live) {
            const uint32_t id = bin->order[idx], r = id / RT3_CTA_THREADS, t = id - r * RT3_CTA_THREADS;
            RT3_ASSERT(r < RT3_RAYS && slot_word_at(sm, r, RT3_F_BOUNCE, t) != RT3_NO_HIT);
            rt3_hit best;
            bvh_closest_hit<true>(S, B, slot_vec_at(sm, r, RT3_F_OX, t), slot_vec_at(sm, r, RT3_F_DX, t), best, visits, tests);
            slot_word_at(sm, r, RT3_F_BEST_T, t) = __float_as_uint(best.t); slot_word_at(sm, r, RT3_F_BEST_PRIM, t) = best.prim;
        }
    }
    __syncthreads(); /* every closest hit is in its slot before the owners shade; nobody is in the pass loop any more */
    if (threadIdx.x == 0) { bin->next_pass = 0u; } /* ordered before the next pass loop by the two barriers in front of it */
    return true;
}

/* The same idea without leaving the warp (no barriers): a warp sorts its own 64 in-flight rays, heavy first, and walks them in two
 * passes of 32. Gains less than the CTA-wide sort (a warp's heavy rays only meet each other) but costs no synchronisation. */
template <bool THREE_CLASSES>
__device__ __forceinline__ void traverse_slots_warp_sorted(const rt3_scene_view& S, const rt3_bvh_view& B, const rt3_smem_view& sm, rt3_bin_scratch* bin,
                                                           uint32_t& visits, uint32_t& tests) {
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, lane_lt = (1u << lane) - 1u;
    static_assert(RT3_RAYS == 2, "the sorted traversal is written for two slots per thread");
    uint16_t* const order = bin->order + warp * (RT3_RAYS * 32u);
    uint32_t inside[RT3_RAYS], heavy[RT3_RAYS], light[RT3_RAYS]; /* THREE_CLASSES: rays that start inside the root box go first, ahead of those that enter it */
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) {
        const bool live = slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT;
        const rt3_vec3 o = slot_vec(sm, r, RT3_F_OX);
        const bool meets = live && ray_meets_box(o, slot_vec(sm, r, RT3_F_DX), bin->root_lo, bin->root_hi);
        const bool in = THREE_CLASSES && meets && o.x >= bin->root_lo[0] && o.x <= bin->root_hi[0] && o.y >= bin->root_lo[1] && o.y <= bin->root_hi[1] &&
                        o.z >= bin->root_lo[2] && o.z <= bin->root_hi[2];
        inside[r] = __ballot_sync(0xffffffffu, in);
        heavy[r] = __ballot_sync(0xffffffffu, meets && !in);
        light[r] = __ballot_sync(0xffffffffu, live && !meets);
    }
    const uint32_t n_inside = (uint32_t) (__popc(inside[0]) + __popc(inside[1])), n_heavy = n_inside + (uint32_t) (__popc(heavy[0]) + __popc(heavy[1])),
                   n_live = n_heavy + (uint32_t) (__popc(light[0]) + __popc(light[1]));
#pragma unroll
    for (int r = 0; r < RT3_RAYS; r++) {
        const uint32_t id = (uint32_t) r * RT3_CTA_THREADS + threadIdx.x;
        if ((inside[r] >> lane) & 1u) { order[(r ? (uint32_t) __popc(inside[0]) : 0u) + (uint32_t) __popc(inside[r] & lane_lt)] = (uint16_t) id; }
        if ((heavy[r] >> lane) & 1u) { order[n_inside + (r ? (uint32_t) __popc(heavy[0]) : 0u) + (uint32_t) __popc(heavy[r] & lane_lt)] = (uint16_t) id; }
        if ((light[r] >> lane) & 1u) { order[n_heavy + (r ? (uint32_t) __popc(light[0]) : 0u) + (uint32_t) __popc(light[r] & lane_lt)] = (uint16_t) id; }
    }
    __syncwarp();
#pragma unroll 1
    for (uint32_t first = 0; first < n_live; first += 32u) {
        const uint32_t idx = first + lane;
        if (idx < n_live) {
            const uint32_t id = order[idx], r = id / RT3_CTA_THREADS, t = id - r * RT3_CTA_THREADS;
            RT3_ASSERT(r < RT3_RAYS && (t >> 5) == warp && slot_word_at(sm, r, RT3_F_BOUNCE, t) != RT3_NO_HIT);
            rt3_hit best;
            bvh_closest_hit<true>(S, B, slot_vec_at(sm, r, RT3_F_OX, t), slot_vec_at(sm, r, RT3_F_DX, t), best, visits, tests);
            slot_word_at(sm, r, RT3_F_BEST_T, t) = __float_as_uint(best.t); slot_word_at(sm, r, RT3_F_BEST_PRIM, t) = best.prim;
        }
    }
    __syncwarp(); /* closest hits are in their slots before the owners shade */
}

/* Adds a thread's traversal counters to the context's (one atomic pair per warp). */
__device__ __forceinline__ void count_accel(uint32_t visits, uint32_t tests, unsigned long long* __restrict__ counters) {
    unsigned long long v = visits, t = tests & ~RT3_BVH_OVERFLOW_BIT;
    const unsigned overflowed = __ballot_sync(0xffffffffu, (tests & RT3_BVH_OVERFLOW_BIT) != 0u);
    for (int off = 16; off > 0; off >>= 1) { v += __shfl_down_sync(0xffffffffu, v, off); t += __shfl_down_sync(0xffffffffu, t, off); }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&counters[2], v); atomicAdd(&counters[3], t);
        if (overflowed) { atomicAdd(&counters[4], (unsigned long long) __popc(overflowed)); }
    }
}

#ifndef RT3_REF_CTAS_PER_SM
#define RT3_REF_CTAS_PER_SM RT3_CTAS_PER_SM
#endif
/* ------------------------------------------------------------------------ *
 * Reference mode: SequentialRenderer.cpp:269-308 (+ AOVs)
 * ------------------------------------------------------------------------ */
template <bool RESIDENT, bool SPHERES_ONLY, bool ACCEL>
__global__ void __launch_bounds__(RT3_CTA_THREADS, RT3_REF_CTAS_PER_SM)
reference_kernel(rt3_scene_view S, rt3_bvh_view B, rt3_camera cam, rt3_kparams P, uint32_t* __restrict__ frame, uint32_t* __restrict__ hit_prim,
                 uint32_t* __restrict__ hit_entity, float* __restrict__ hit_t, unsigned long long* __restrict__ counters) {
    constexpr int R = RT3_REF_RAYS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const rt3_smem_view sm = smem_view<RESIDENT, ACCEL, RT3_MASK_BYTES_FOR(RT3_REF_RAYS)>(smem_raw);
    scene_prologue<RESIDENT>(sm);
    uint32_t phase = 0u;

    const rt3_vec3 origin = v3(cam.origin[0], cam.origin[1], cam.origin[2]);
    const rt3_vec3 hor = v3(cam.horizontal[0], cam.horizontal[1], cam.horizontal[2]);
    const rt3_vec3 ver = v3(cam.vertical[0], cam.vertical[1], cam.vertical[2]);
    const rt3_vec3 llc = v3(cam.lower_left_corner[0], cam.lower_left_corner[1], cam.lower_left_corner[2]);

    rt3_vec3 o[R], d[R], dn[R];
    bool live[R];
    rt3_hit best[R];
    size_t pix[R];
    const unsigned long long cta_first = (unsigned long long) blockIdx.x * (RT3_CTA_THREADS * R);
#pragma unroll
    for (int r = 0; r < R; r++) {
        unsigned long long p = cta_first + (unsigned long long) r * RT3_CTA_THREADS + threadIdx.x;
        live[r] = p < P.n_pixels;
        if (!live[r]) { p = 0; }
        uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
        uint32_t y = owned_row_to_global(P, local_row);
        pix[r] = (size_t) y * P.width + x;
        /* SequentialRenderer.cpp:289-293: the divides are written in double there */
        float u = (float) ((double) (float) x / ((double) (float) P.width - 1.0));
        float v = (float) ((double) (float) (P.height - 1 - y) / ((double) (float) P.height - 1.0));
        o[r] = origin;
        d[r] = ((llc + u * hor) + v * ver) - origin;
        dn[r] = normalize3(d[r]);
    }
    uint32_t visits = 0, tests = 0;
    if (ACCEL) {
#pragma unroll
        for (int r = 0; r < R; r++) {
            best[r].t = __int_as_float(0x7f800000); best[r].prim = RT3_NO_HIT;
            if (live[r]) { bvh_closest_hit<false>(S, B, o[r], d[r], best[r], visits, tests); }
        }
    } else {
        sweep_scene<false, RESIDENT, SPHERES_ONLY, R>(S, sm, phase, o, d, dn, live, best);
    }
    unsigned long long rays = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        if (!live[r]) { continue; }
        rays++;
        rt3_vec3 col;
        uint32_t ent = RT3_NO_HIT;
        if (best[r].prim == RT3_NO_HIT) {
            /* sky, SequentialRenderer.cpp:105-107 */
            float len = sqrtf(dot3(d[r], d[r]));
            float uy = d[r].y / len;
            float t = (float) (0.5 * ((double) uy + 1.0));
            float a = 1.0f - t;
            col = v3(a * 1.0f + t * 0.5f, a * 1.0f + t * 0.7f, a * 1.0f + t * 1.0f);
        } else {
            float4 c = __ldg(&S.prim_color[best[r].prim]);
            col = v3(c.x, c.y, c.z);
            ent = __ldg(&S.prim_entity[best[r].prim]);
        }
        frame[pix[r]] = pack_rgb(col);
        if (hit_prim) { hit_prim[pix[r]] = best[r].prim; }
        if (hit_entity) { hit_entity[pix[r]] = ent; }
        if (hit_t) { hit_t[pix[r]] = best[r].t; }
    }
    /* ray count: one atomic per warp */
    for (int off = 16; off > 0; off >>= 1) { rays += __shfl_down_sync(0xffffffffu, rays, off); }
    if ((threadIdx.x & 31) == 0 && rays) { atomicAdd(&counters[1], rays); }
    if (ACCEL) { count_accel(visits, tests, counters); }
}

/* ------------------------------------------------------------------------ *
 * Path tracer
 * ------------------------------------------------------------------------ */

/* Uniform point on the unit sphere: z = 1 - 2 xi1, phi = 2 pi xi2. */
__device__ __forceinline__ rt3_vec3 unit_vector(float xi1, float xi2) {
    float z = 1.0f - 2.0f * xi1;
    float rr = 1.0f - z * z;
    rr = sqrtf(rr < 0.0f ? 0.0f : rr);
    float sn, cs;
    rt3_sincos_2pi(xi2, &sn, &cs);
    return v3(rr * cs, rr * sn, z);
}

__device__ __forceinline__ unsigned long long to_fixed(float c) {
    if (!(c > 0.0f)) { return 0ull; }
    if (c > 1048576.0f) { c = 1048576.0f; }
    return (unsigned long long) (c * RT3_ACC_SCALE + 0.5f);
}

/* A warp's current chunk of path items [cur, end) out of the global counter,
 * with the (pixel, sample) of its first item so that per-item decoding needs
 * 32-bit arithmetic only. All fields are warp-uniform. */
struct rt3_chunk {
    unsigned long long cur, end, start;
    uint32_t pixel0, sample0; /* item `start` = (pixel0, sample0) */
    bool dry;                 /* the global counter is exhausted */
    bool beam_ok;             /* BEAM kernels: the chunk has a candidate list for its primary rays (rt3_beam) ... */
    uint32_t beam_candidates; /* ... of this many primitives */
};
/* (`start` doubles as the warp's last reading of the global counter: the value its previous claim returned.) */

/* Items a warp takes from the global counter at a time: RT3_ITEM_CHUNK while there is plenty left, shrinking with
 * what remains (guided self-scheduling) so that the warps run dry together -- with the frame split over 8 GPUs
 * a kernel is only ~17 ms long and a fixed chunk of 256 items is a visible tail. `seen` is a stale reading of the
 * counter (what the warp's previous claim returned: no extra load); any value is correct, it only steers the size. */
__device__ __forceinline__ unsigned long long chunk_size(unsigned long long seen, const rt3_kparams& P) {
    const unsigned long long left = seen < P.n_items ? P.n_items - seen : 0ull;
    const uint32_t claimers = gridDim.x * (RT3_CTA_THREADS / 32) * 2u;
    if (left >= (unsigned long long) RT3_ITEM_CHUNK * claimers) { return RT3_ITEM_CHUNK; } /* the common case: no division */
    const uint32_t share = (uint32_t) left / claimers;                                      /* left < 256 * claimers < 2^32 */
    return share <= RT3_ITEM_CHUNK_MIN ? RT3_ITEM_CHUNK_MIN : share;
}

/* Warp-cooperative claim of one path item per requesting lane. Items are
 * item = pixel * spp + sample over this partition's compact pixel list. */
__device__ __forceinline__ bool claim_item(bool want, rt3_chunk& c, const rt3_kparams& P, unsigned long long* next_item,
                                           uint32_t& pixel, uint32_t& sample) {
    const unsigned lane = threadIdx.x & 31u;
    unsigned m = __ballot_sync(0xffffffffu, want);
    int n = __popc(m);
    int rank = __popc(m & ((1u << lane) - 1u));
    bool got = false;
    while (n > 0 && !c.dry) {
        if (c.cur == c.end) {
            unsigned long long v = 0, size = 0;
            if (lane == 0) {
                size = chunk_size(c.start, P);
                v = atomicAdd(next_item, size);
            }
            v = __shfl_sync(0xffffffffu, v, 0);
            size = __shfl_sync(0xffffffffu, size, 0);
            if (v >= P.n_items) { c.dry = true; break; }
            c.cur = c.start = v;
            c.end = v + size < P.n_items ? v + size : P.n_items;
            unsigned long long p0 = v / P.spp; /* one 64-bit divide per chunk */
            c.pixel0 = (uint32_t) p0;
            c.sample0 = (uint32_t) (v - p0 * P.spp);
        }
        unsigned long long avail = c.end - c.cur;
        int take = (unsigned long long) n < avail ? n : (int) avail;
        if (want && !got && rank >= 0 && rank < take) {
            uint32_t k = (uint32_t) (c.cur - c.start) + (uint32_t) rank + c.sample0; /* < spp + chunk */
            uint32_t dp = k / P.spp;
            pixel = c.pixel0 + dp;
            sample = k - dp * P.spp;
            got = true;
        }
        rank -= take;
        c.cur += (unsigned long long) take;
        n -= take;
    }
    return got;
}

/* One path slot while it is in registers: the ray being traced, its throughput and its RNG key. */
struct rt3_path {
    rt3_vec3 o, d, thr;
    uint32_t key, bounce, pix; /* bounce == RT3_NO_HIT: the slot is free */
};

struct rt3_cam_view {
    rt3_vec3 origin, hor, ver, llc, lens_u, lens_v;
    float lens_radius, wm1, hm1;
};

/* Primary ray of path item (compact pixel p, sample): pixel jitter, thin lens. */
__device__ __forceinline__ void start_path(rt3_path& s, const rt3_cam_view& C, const rt3_kparams& P, uint32_t p, uint32_t sample) {
    uint32_t local_row = p / P.width, x = p - local_row * P.width;
    uint32_t y = owned_row_to_global(P, local_row);
    uint32_t pixel_index = y * P.width + x;
    s.pix = pixel_index;
    uint32_t k = rt3_path_key(pixel_index, P.first_sample + sample, P.seed);
    s.key = k;
    float jx = 0.0f, jy = 0.0f;
    if (!(P.flags & RT3_FLAG_NO_JITTER)) { jx = rt3_draw(k, RT3_DIM_JITTER_X); jy = rt3_draw(k, RT3_DIM_JITTER_Y); }
    float u = ((float) x + jx) / C.wm1;
    float v = ((float) (P.height - 1 - y) + jy) / C.hm1;
    rt3_vec3 org = C.origin;
    rt3_vec3 dir = ((C.llc + u * C.hor) + v * C.ver) - org;
    if (C.lens_radius > 0.0f) {
        float rad = sqrtf(rt3_draw(k, RT3_DIM_LENS_R));
        float sn, cs;
        rt3_sincos_2pi(rt3_draw(k, RT3_DIM_LENS_PHI), &sn, &cs);
        float lx = C.lens_radius * (rad * cs), ly = C.lens_radius * (rad * sn);
        rt3_vec3 off = lx * C.lens_u + ly * C.lens_v;
        org = org + off;
        dir = dir - off;
    }
    s.o = org;
    s.d = normalize3(dir);
    s.thr = v3(1.0f, 1.0f, 1.0f);
    s.bounce = 0;
}

/* Radiance of a path that left the scene: throughput times the reference's sky (SequentialRenderer.cpp:105-107, unit direction). */
__device__ __forceinline__ rt3_vec3 shade_miss(rt3_vec3 thr, rt3_vec3 dr, const rt3_kparams& P) {
    float t = 0.5f * (dr.y + 1.0f);
    float a = 1.0f - t;
    rt3_vec3 L = thr * v3(a * 1.0f + t * 0.5f, a * 1.0f + t * 0.7f, a * 1.0f + t * 1.0f);
    if (P.flags & RT3_FLAG_UNIFORM_SKY) { L = thr; } /* white furnace */
    return L;
}

/* Adds a finished path's radiance to its pixel's fixed-point accumulators. */
__device__ __forceinline__ void add_radiance(unsigned long long* __restrict__ accum, uint32_t pix, rt3_vec3 L, const rt3_kparams& P) {
    unsigned long long qx = to_fixed(L.x), qy = to_fixed(L.y), qz = to_fixed(L.z);
    RT3_ASSERT(pix < P.width * P.height);
    unsigned long long* acc = accum + 3 * (size_t) pix;
    if (qx) { atomicAdd(acc + 0, qx); }
    if (qy) { atomicAdd(acc + 1, qy); }
    if (qz) { atomicAdd(acc + 2, qz); }
}

/* Shades the closest hit `best` of a live path: miss -> sky * throughput, hit -> scatter
 * (Lambertian, metal, dielectric; SURVEY.md appendix C). A finished path adds its radiance to the
 * pixel's fixed-point accumulators and frees the slot. */
__device__ __forceinline__ void shade_path(rt3_path& s, const rt3_hit& best, const rt3_scene_view& S, const rt3_kparams& P,
                                           unsigned long long* __restrict__ accum) {
    bool done = false;
    rt3_vec3 L = v3(0.0f, 0.0f, 0.0f);
    const rt3_vec3 dr = s.d;
    if (best.prim == RT3_NO_HIT) {
        L = shade_miss(s.thr, dr, P);
        done = true;
    } else {
        const uint32_t prim = best.prim;
        RT3_ASSERT(prim < S.n_prims);
        rt3_vec3 hp = s.o + best.t * dr;
        rt3_vec3 outward;
        if (prim < S.n_faces) {
            float4 fn = __ldg(&S.face_rec[4 * (size_t) prim]);
            outward = v3(fn.x, fn.y, fn.z);
        } else {
            float4 sp = __ldg(&S.spheres[prim - S.n_faces]);
            rt3_vec3 pc = hp - v3(sp.x, sp.y, sp.z);
            outward = v3(pc.x / sp.w, pc.y / sp.w, pc.z / sp.w);
        }
        const bool front = dot3(dr, outward) < 0.0f;
        const rt3_vec3 n = front ? outward : -outward;
        uint32_t kind = RT3_MAT_LAMBERTIAN;
        rt3_vec3 albedo;
        float fuzz = 0.0f, ior = 1.0f;
        const uint32_t mi = __ldg(&S.prim_material[prim]);
        if (mi == RT3_NO_HIT) {
            float4 c = __ldg(&S.prim_color[prim]);
            albedo = v3(c.x, c.y, c.z);
        } else {
            float4 m0 = __ldg(&S.materials[2 * mi]), m1 = __ldg(&S.materials[2 * mi + 1]);
            kind = __float_as_uint(m0.x);
            albedo = v3(m0.y, m0.z, m0.w);
            fuzz = m1.x; ior = m1.y;
        }
        const uint32_t dim = RT3_DIM_BOUNCE0 + RT3_DIMS_PER_BOUNCE * s.bounce;
        const uint32_t k = s.key;
        rt3_vec3 nd;
        /* every material's first draws are dims +0 and +1 (the oracle's layout); drawn once, ahead of the
         * material branches, so that a warp with mixed materials runs the hash and the sincos polynomial once */
        const float xi0 = rt3_draw(k, dim + 0), xi1 = rt3_draw(k, dim + 1);
        const rt3_vec3 uv = unit_vector(xi0, xi1);
        if (kind == RT3_MAT_LAMBERTIAN) {
            nd = n + uv;
            if (fabsf(nd.x) < 1e-8f && fabsf(nd.y) < 1e-8f && fabsf(nd.z) < 1e-8f) { nd = n; }
            s.thr = s.thr * albedo;
        } else if (kind == RT3_MAT_METAL) {
            float dnn = dot3(dr, n);
            nd = dr - (2.0f * dnn) * n;
            float fz = fuzz < 1.0f ? fuzz : 1.0f;
            if (fz > 0.0f) {
                float a = rt3_draw(k, dim + 2), b = rt3_draw(k, dim + 3), c = rt3_draw(k, dim + 4);
                float mx = a < b ? b : a;
                mx = mx < c ? c : mx;
                nd = nd + (fz * mx) * uv;
            }
            if (!(dot3(nd, n) > 0.0f)) { done = true; }
            s.thr = s.thr * albedo;
        } else {
            float ratio = front ? (1.0f / ior) : ior;
            float cs = -dot3(dr, n);
            cs = cs < 1.0f ? cs : 1.0f;
            float s2 = 1.0f - cs * cs;
            float sn = sqrtf(s2 < 0.0f ? 0.0f : s2);
            bool cannot_refract = ratio * sn > 1.0f;
            float r0 = (1.0f - ratio) / (1.0f + ratio);
            r0 = r0 * r0;
            float w = 1.0f - cs;
            float w2 = w * w;
            float schlick = r0 + (1.0f - r0) * ((w2 * w2) * w);
            if (cannot_refract || schlick > xi0) {
                float dnn = dot3(dr, n);
                nd = dr - (2.0f * dnn) * n;
            } else {
                rt3_vec3 perp = ratio * (dr + cs * n);
                float kk = 1.0f - dot3(perp, perp);
                rt3_vec3 par = (-sqrtf(fabsf(kk))) * n;
                nd = perp + par;
            }
        }
        if (!done) {
            s.o = hp;
            s.d = normalize3(nd);
            s.bounce++;
            if (s.bounce >= P.max_depth) { done = true; } /* depth exhausted: radiance 0 */
        }
    }
    if (done) {
        add_radiance(accum, s.pix, L, P);
        s.bounce = RT3_NO_HIT;
    }
}

/* ---- primary rays through a candidate list (BEAM kernels: resident sphere scenes) -------------------------------------
 * A third of all ray segments of BASELINE C2 are primary rays, and the primary rays of one pixel are nearly the same ray:
 * they leave the lens (radius L around the camera origin O) and pass through the pixel's footprint on the focus plane. A
 * warp claims its path items a chunk at a time, and a chunk of 256 items of a 500-spp frame lies in one or two pixels. So
 * once per CHUNK the warp tests every primitive against the chunk's BEAM -- everything a primary ray of these pixels can
 * reach -- and keeps the candidates as a bit mask; the primary ray of each item then runs the exact tests of the
 * candidates only (a handful), in ascending order like the sweep's drain, and is shaded before the slot sees its first
 * sweep. A path thus occupies a slot for its bounce segments only: 1.75 instead of 2.75 sweeps per path on C2.
 *
 * The beam. Item (x, y, sample) aims at T = llc + u hor + v ver with u in [x, x + 1) / (W - 1), v likewise, from O + off,
 * |off| <= L' = L (|lens_u| + |lens_v|). With T0 the centre of the chunk's pixel range, D = T0 - O and
 * delta >= |T - T0|, a point of the ray is P(s) = O + off + s (T - O - off) = Q(s) + (1 - s) off + s (T - T0), where
 * Q(s) = O + s D is the central ray, hence |P(s) - Q(s)| <= L' + s k with k = L' + delta. The exact sphere test can only
 * report a sphere whose centre C lies within Re of the ray's line (Re^2 = r^2 + slack (|C|^2 + r^2 + |o|^2): the
 * conservativeness argument of the level-1 filter, rt3_device.cuh / DESIGN.md 3.1). So if the ray reaches the sphere at
 * parameter s then |Q(s) - C| <= Re + L' + s k; because |Q(s) - C| >= |s - s*| |D| (s* = the parameter of C's projection on
 * the central line), s <= s_hi = (max(s*, 0) |D| + Re + L') / (|D| - k), and C is within Re + L' + s_hi k of the central
 * line. Primitives that fail this test cannot be reported for any item of the chunk; the others are candidates. All of it
 * is evaluated with generous roundings (the comparison carries 2^-20 |C - O|^2 and 1 + 1e-5): a wrong candidate costs one
 * exact test, a missing one would be a wrong frame. Chunks that span rows or many pixels, beams with too many
 * candidates and degenerate cameras fall back to the sweep (ok = 0): their primary rays are traced like every other ray. */
#define RT3_BEAM_WORDS (RT3_CONST_PRIMS / 32)
#ifndef RT3_BEAM_MAX_PIXELS
#define RT3_BEAM_MAX_PIXELS 64u
#endif
#ifndef RT3_BEAM_MAX_CANDIDATES
#define RT3_BEAM_MAX_CANDIDATES 48u
#endif
#ifndef RT3_BEAM_MIN_BATCH
#define RT3_BEAM_MIN_BATCH 8u /* a further regeneration batch of a round runs only for at least this many free slots (a batch turn costs the warp about as much
                               * as sweeping nine slots); what stays free is filled by the first batch of the next round. C2, call AK
                               * (profiles/r02ak_variants.jsonl): 1: 116.12 ms, 4: 116.02, 8: 115.66, 16: 116.60 */
#endif
#ifndef RT3_BEAM_EARLY_OUT
#define RT3_BEAM_EARLY_OUT 1 /* exact_sphere_path_coherent in the candidate tests of the sweep's BEAM kernel */
#endif
#ifndef RT3_BEAM_BATCHES
#define RT3_BEAM_BATCHES 4u /* regeneration batches per round at most (the first takes up to 32 of the warp's free slots, the next ones the rest and
                             * the slots of paths that ended with their primary ray; what is still free after that waits for the next round).
                             * C2, call AD: 1 batch 128.3 ms, 2: 117.8, 3: 117.2, 4: 116.9 (plain sweep 136.2) */
#endif
struct rt3_beam {                      /* one per warp, in shared memory behind the path slots */
    uint16_t list[64];                 /* candidates of the warp's current chunk, ascending primitive ids (RT3_BEAM_MAX_CANDIDATES <= 64 used) */
};
static_assert(RT3_BEAM_MAX_CANDIDATES <= 64u && RT3_CONST_PRIMS <= 0x10000, "candidate ids are 16 bits wide, the list holds 64");
static_assert(sizeof(rt3_beam) == 128, "one 128-byte line per warp");
#define RT3_BEAM_BYTES ((RT3_CTA_THREADS / 32) * 128)

/* Approximate square root and reciprocal (one MUFU each, 2^-22 relative): the beam test carries far larger safety factors, and the
 * IEEE versions would add 3 KB of code to a kernel whose loop has to stay inside the 32 KB instruction cache. */
__device__ __forceinline__ float beam_sqrt(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float beam_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

/* The whole warp: candidate list of the chunk `c` has just claimed (spheres only). */
__device__ __forceinline__ void beam_for_chunk(const rt3_scene_view& S, const rt3_cam_view& C, const rt3_kparams& P, rt3_chunk& c, rt3_beam* beam) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t p_first = c.pixel0, p_last = c.pixel0 + ((uint32_t) (c.end - 1ull - c.start) + c.sample0) / P.spp; /* 32-bit: < spp + chunk */
    const uint32_t row = p_first / P.width;
    const uint32_t xa = p_first - row * P.width, xb = p_last - row * P.width;
    bool ok = p_last / P.width == row && xb - xa < RT3_BEAM_MAX_PIXELS && S.n_faces == 0u && S.n_prims <= (uint32_t) RT3_CONST_PRIMS;
    const uint32_t y = owned_row_to_global(P, row);
    /* the (u, v) range of the chunk's pixels, jitter included, and its centre */
    const float iw = beam_rcp(C.wm1), ih = beam_rcp(C.hm1);
    const float u0 = (float) xa * iw, u1 = ((float) xb + 1.0f) * iw;
    const float v0 = (float) (P.height - 1u - y) * ih, v1 = ((float) (P.height - 1u - y) + 1.0f) * ih;
    const float um = 0.5f * (u0 + u1), vm = 0.5f * (v0 + v1);
    const rt3_vec3 D = ((C.llc + um * C.hor) + vm * C.ver) - C.origin;
    const float len_hor = beam_sqrt(dot3(C.hor, C.hor)), len_ver = beam_sqrt(dot3(C.ver, C.ver)), len_o = beam_sqrt(dot3(C.origin, C.origin));
    const float tiny = 4.76837158203125e-07f * ((len_hor + len_ver) + (beam_sqrt(dot3(C.llc, C.llc)) + len_o)); /* 2^-21: roundings of T and of o + off */
    const float delta = (0.5f * (u1 - u0) * len_hor + 0.5f * (v1 - v0) * len_ver) * 1.001f + tiny;
    const float lens = C.lens_radius > 0.0f ? C.lens_radius * (beam_sqrt(dot3(C.lens_u, C.lens_u)) + beam_sqrt(dot3(C.lens_v, C.lens_v))) * 1.001f + tiny : tiny;
    const float k = lens + delta;
    const float dd = dot3(D, D), len_d = beam_sqrt(dd);
    ok = ok && len_d > 4.0f * k && len_d < 1e18f && k < 1e18f; /* false for NaN too */
    const float inv_dd = beam_rcp(dd), inv_reach = beam_rcp(len_d - k);
    const float o_max = len_o + lens, o_slack = RT3_FILTER_SLACK * (o_max * o_max);
    const uint32_t n_words = (S.n_prims + 31u) / 32u;
    uint32_t n_candidates = 0;
#pragma unroll 1
    for (uint32_t w = 0; w < n_words; w++) {
        const uint32_t prim = w * 32u + lane;
        bool candidate = false;
        if (ok && prim < S.n_prims) {
            const float4 sp = __ldg(&S.spheres[prim]);
            const rt3_vec3 ctr = v3(sp.x, sp.y, sp.z), co = ctr - C.origin;
            const float r2 = sp.w * sp.w;
            const float re = beam_sqrt((r2 + RT3_FILTER_SLACK * (dot3(ctr, ctr) + r2) + o_slack) * 1.0001f);
            const float proj = dot3(co, D), co2 = dot3(co, co);
            const float s_star = proj * inv_dd;
            const float dist2 = co2 - s_star * proj;
            const float s_hi = (fmaxf(s_star, 0.0f) * len_d + re + lens) * inv_reach;
            const float reach = (re + lens + s_hi * k) * 1.0001f;
            candidate = !(dist2 > reach * reach + 1.9073486328125e-06f * co2); /* 2^-19 |C - O|^2 for the roundings; a NaN anywhere keeps the primitive */
        }
        const uint32_t m = __ballot_sync(0xffffffffu, candidate);
        const uint32_t at = n_candidates + (uint32_t) __popc(m & ((1u << lane) - 1u));
        if (candidate && at < RT3_BEAM_MAX_CANDIDATES) { beam->list[at] = (uint16_t) prim; } /* ascending: words in order, lanes in order */
        n_candidates += (uint32_t) __popc(m);
    }
    ok = ok && n_candidates <= RT3_BEAM_MAX_CANDIDATES;
    /* (no conditional around the votes above and no __syncwarp here: either makes ptxas give up the uniform loads of the sweep, see
     * tests/test_sass_evidence.py; the caller synchronises the warp before the list is read) */
    c.beam_ok = ok; c.beam_candidates = n_candidates;
}

/* ---- the same through the hierarchy (ACCEL + BEAM kernels: any scene rendered with RT3_FLAG_BVH) -----------------------
 * The chunk's beam walks the two trees once, the whole warp at a time and level by level: the lanes take one node of the
 * current level each, test both child boxes against the beam and append the children that meet it to the next level
 * (internal nodes) or to the candidate list (leaves). A ray can only be reported a primitive whose (host-widened) box,
 * grown by ray_margin |o|, it crosses -- that is the hierarchy's own contract, rt3_bvh.cuh -- so a box the beam misses
 * holds no primitive that any primary ray of the chunk could be reported. The box is tested through its bounding sphere
 * (centre, half diagonal + sqrt(3) ray_margin o_max) with the inequality of beam_for_chunk above; NaNs and infinities keep
 * the box. Levels wider than RT3_ABEAM_LEVEL nodes and lists longer than RT3_ABEAM_MAX_CANDIDATES give the chunk up (ok = 0: its primary
 * rays walk the hierarchy like every other ray). The primary rays then run the exact tests of the candidates with the
 * hierarchy's tie rule (lower primitive id), whatever the order of the list. */
#ifndef RT3_ABEAM_MAX_PIXELS
#define RT3_ABEAM_MAX_PIXELS 16u
#endif
#ifndef RT3_ABEAM_MAX_CANDIDATES
#define RT3_ABEAM_MAX_CANDIDATES 192u    /* a beam does not stop at the first hit: on BASELINE C5 (10^6 spheres, four pixels per chunk) it meets 56 primitives on
                                          * average and up to 150 (CPU model of the walk); 128 exact tests at full lanes still cost less than 129 node visits at a third */
#endif
#ifndef RT3_ABEAM_BATCHES
#define RT3_ABEAM_BATCHES 16u            /* regeneration batches per round at most: a scene of depth 1 (C5) never fills a slot, and every round pays RT3_RAYS idle slot turns */
#endif
#define RT3_ABEAM_LEVEL 192u             /* nodes per level of the walk: C5 reaches 100 on average, 153 at most in the same model */
struct __align__(16) rt3_abeam {          /* one per warp, in shared memory behind the exchange area */
    uint32_t list[RT3_ABEAM_MAX_CANDIDATES]; /* candidate primitives of the warp's current chunk (global ids, no particular order) */
};
#define RT3_ABEAM_EXCHANGE_BYTES (12 * RT3_CTA_THREADS * 4) /* the hierarchy kernels have no survivor masks to alias the exchange area on */
#define RT3_ABEAM_BYTES (RT3_ABEAM_EXCHANGE_BYTES + (RT3_CTA_THREADS / 32) * sizeof(rt3_abeam))
static_assert(2u * RT3_ABEAM_LEVEL == 12u * 32u, "the two levels of the walk live in the warp's 12 x 32 words of the exchange area, which is idle while a chunk is claimed");
/* word i of level `which` of this warp's walk (`exchange` points at the warp's first column) */
__device__ __forceinline__ uint32_t& abeam_level(uint32_t* exchange, uint32_t which, uint32_t i) {
    const uint32_t w = which * RT3_ABEAM_LEVEL + i;
    return exchange[(w >> 5) * RT3_CTA_THREADS + (w & 31u)];
}

__device__ __forceinline__ void beam_for_chunk_bvh(const rt3_bvh_view& B, const rt3_cam_view& C, const rt3_kparams& P, rt3_chunk& c, rt3_abeam* ab,
                                                   uint32_t* exchange, uint32_t& visits) {
    const uint32_t lane = threadIdx.x & 31u, lane_lt = (1u << lane) - 1u;
    const uint32_t p_first = c.pixel0, p_last = c.pixel0 + ((uint32_t) (c.end - 1ull - c.start) + c.sample0) / P.spp;
    const uint32_t row = p_first / P.width;
    const uint32_t xa = p_first - row * P.width, xb = p_last - row * P.width;
    bool ok = p_last / P.width == row && xb - xa < RT3_ABEAM_MAX_PIXELS;
    const uint32_t y = owned_row_to_global(P, row);
    /* the beam of the chunk's pixels: as in beam_for_chunk */
    const float iw = beam_rcp(C.wm1), ih = beam_rcp(C.hm1);
    const float u0 = (float) xa * iw, u1 = ((float) xb + 1.0f) * iw;
    const float v0 = (float) (P.height - 1u - y) * ih, v1 = ((float) (P.height - 1u - y) + 1.0f) * ih;
    const float um = 0.5f * (u0 + u1), vm = 0.5f * (v0 + v1);
    const rt3_vec3 D = ((C.llc + um * C.hor) + vm * C.ver) - C.origin;
    const float len_hor = beam_sqrt(dot3(C.hor, C.hor)), len_ver = beam_sqrt(dot3(C.ver, C.ver)), len_o = beam_sqrt(dot3(C.origin, C.origin));
    const float tiny = 4.76837158203125e-07f * ((len_hor + len_ver) + (beam_sqrt(dot3(C.llc, C.llc)) + len_o));
    const float delta = (0.5f * (u1 - u0) * len_hor + 0.5f * (v1 - v0) * len_ver) * 1.001f + tiny;
    const float lens = C.lens_radius > 0.0f ? C.lens_radius * (beam_sqrt(dot3(C.lens_u, C.lens_u)) + beam_sqrt(dot3(C.lens_v, C.lens_v))) * 1.001f + tiny : tiny;
    const float k = lens + delta;
    const float dd = dot3(D, D), len_d = beam_sqrt(dd);
    ok = ok && len_d > 4.0f * k && len_d < 1e18f && k < 1e18f; /* false for NaN too */
    const float inv_dd = beam_rcp(dd), inv_reach = beam_rcp(len_d - k);
    const float o_max = len_o + lens;
    uint32_t n_candidates = 0;
#pragma unroll 1
    for (int which = 0; which < 2; which++) {
        const rt3_bvh_tree T = B.tree[which];
        if (!ok || T.n_prims == 0u) { continue; } /* warp-uniform, like everything that guards a vote below */
        if (T.root < 0) { /* a tree of one primitive */
            if (lane == 0 && n_candidates < RT3_ABEAM_MAX_CANDIDATES) { ab->list[n_candidates] = (uint32_t) ~T.root; }
            n_candidates++;
            continue;
        }
        const float grow = 1.7320508f * T.ray_margin * o_max * 1.0001f + tiny; /* the per-ray widening of a box, at its corners */
        uint32_t n_cur = 1u, cur = 0u;
        if (lane == 0) { abeam_level(exchange, 0u, 0u) = (uint32_t) T.root; }
        __syncwarp();
#pragma unroll 1
        while (n_cur != 0u) {
            uint32_t n_next = 0u;
#pragma unroll 1
            for (uint32_t base = 0; base < n_cur; base += 32u) {
                bool meets[2] = { false, false };
                int32_t ref[2] = { 0, 0 };
                if (base + lane < n_cur) {
                    const int32_t node = (int32_t) abeam_level(exchange, cur, base + lane);
                    RT3_ASSERT(node >= 0 && (uint32_t) node + 2u <= B.tree[0].n_prims + B.tree[1].n_prims);
                    visits++;
                    const float4 n0 = __ldg(&B.nodes[4 * node + 0]), n1 = __ldg(&B.nodes[4 * node + 1]), n2 = __ldg(&B.nodes[4 * node + 2]),
                                 n3 = __ldg(&B.nodes[4 * node + 3]);
                    const float lo[2][3] = { { n0.x, n0.y, n0.z }, { n1.z, n1.w, n2.x } }, hi[2][3] = { { n0.w, n1.x, n1.y }, { n2.y, n2.z, n2.w } };
                    ref[0] = __float_as_int(n3.x); ref[1] = __float_as_int(n3.y);
#pragma unroll
                    for (int ch = 0; ch < 2; ch++) {
                        const rt3_vec3 ctr = v3(0.5f * lo[ch][0] + 0.5f * hi[ch][0], 0.5f * lo[ch][1] + 0.5f * hi[ch][1], 0.5f * lo[ch][2] + 0.5f * hi[ch][2]);
                        const rt3_vec3 half = v3(0.5f * hi[ch][0] - 0.5f * lo[ch][0], 0.5f * hi[ch][1] - 0.5f * lo[ch][1], 0.5f * hi[ch][2] - 0.5f * lo[ch][2]);
                        const float rho = beam_sqrt(dot3(half, half));
                        /* + 2^-21 (|centre| + rho): the roundings of the centre and of centre - O */
                        const float re = (rho + grow) * 1.0001f + 4.76837158203125e-07f * (((fabsf(ctr.x) + fabsf(ctr.y)) + fabsf(ctr.z)) + rho);
                        const rt3_vec3 co = ctr - C.origin;
                        const float proj = dot3(co, D), co2 = dot3(co, co);
                        const float s_star = proj * inv_dd;
                        const float dist2 = co2 - s_star * proj;
                        const float s_hi = (fmaxf(s_star, 0.0f) * len_d + re + lens) * inv_reach;
                        const float reach = (re + lens + s_hi * k) * 1.0001f;
                        meets[ch] = !(dist2 > reach * reach + 1.9073486328125e-06f * co2); /* a NaN anywhere keeps the box */
                    }
                }
#pragma unroll
                for (int ch = 0; ch < 2; ch++) {
                    const uint32_t m_in = __ballot_sync(0xffffffffu, meets[ch] && ref[ch] >= 0), m_lf = __ballot_sync(0xffffffffu, meets[ch] && ref[ch] < 0);
                    const uint32_t at_in = n_next + (uint32_t) __popc(m_in & lane_lt), at_lf = n_candidates + (uint32_t) __popc(m_lf & lane_lt);
                    if (meets[ch] && ref[ch] >= 0 && at_in < RT3_ABEAM_LEVEL) { abeam_level(exchange, cur ^ 1u, at_in) = (uint32_t) ref[ch]; }
                    if (meets[ch] && ref[ch] < 0 && at_lf < RT3_ABEAM_MAX_CANDIDATES) { ab->list[at_lf] = (uint32_t) ~ref[ch]; }
                    n_next += (uint32_t) __popc(m_in); n_candidates += (uint32_t) __popc(m_lf);
                }
            }
            __syncwarp();
            if (n_next > RT3_ABEAM_LEVEL || n_candidates > RT3_ABEAM_MAX_CANDIDATES) { ok = false; n_next = 0u; }
            cur ^= 1u; n_cur = n_next;
        }
    }
    ok = ok && n_candidates <= RT3_ABEAM_MAX_CANDIDATES;
    c.beam_ok = ok; c.beam_candidates = n_candidates;
}

/* Closest hit of a primary ray among the candidates the beam's walk collected: the leaf tests of bvh_closest_hit (path mode). Four
 * candidates at a time when they are all spheres -- their records are loaded together, so that a lane waits for one load instead of four
 * in a row (the tests of one ray depend on each other through `best` only) -- and one by one otherwise. */
#ifndef RT3_ABEAM_GROUP
#define RT3_ABEAM_GROUP 1
#endif
#ifndef RT3_ABEAM_EARLY_OUT
#define RT3_ABEAM_EARLY_OUT 1 /* the lanes test the same sphere: leave at the discriminant when it is negative (exact_sphere_path_coherent) */
#endif
#if RT3_ABEAM_EARLY_OUT
#define RT3_ABEAM_SPHERE_TEST exact_sphere_path_coherent<false>
#else
#define RT3_ABEAM_SPHERE_TEST exact_sphere_path<false>
#endif
__device__ __forceinline__ void beam_closest_hit_bvh(const rt3_scene_view& S, const rt3_abeam* ab, uint32_t n_candidates, bool active, rt3_vec3 o, rt3_vec3 d, rt3_hit& best) {
    best.t = __int_as_float(0x7f800000);
    best.prim = RT3_NO_HIT;
#pragma unroll 1
    for (uint32_t i = 0; i < n_candidates;) { /* i stays a multiple of four up to the last group */
        const uint32_t g = n_candidates - i < 4u ? n_candidates - i : 4u;
        bool done = false;
#if RT3_ABEAM_GROUP
        if (g == 4u) {
            const uint4 p = *reinterpret_cast<const uint4*>(&ab->list[i]); /* warp-uniform */
            RT3_ASSERT(p.x < S.n_prims && p.y < S.n_prims && p.z < S.n_prims && p.w < S.n_prims);
            if (min(min(p.x, p.y), min(p.z, p.w)) >= S.n_faces) {
                const float4 s0 = __ldg(&S.spheres[p.x - S.n_faces]), s1 = __ldg(&S.spheres[p.y - S.n_faces]), s2 = __ldg(&S.spheres[p.z - S.n_faces]),
                             s3 = __ldg(&S.spheres[p.w - S.n_faces]);
                if (active) {
                    RT3_ABEAM_SPHERE_TEST(p.x, s0, o, d, best); RT3_ABEAM_SPHERE_TEST(p.y, s1, o, d, best);
                    RT3_ABEAM_SPHERE_TEST(p.z, s2, o, d, best); RT3_ABEAM_SPHERE_TEST(p.w, s3, o, d, best);
                }
                done = true;
            }
        }
#endif
        if (!done) {
#pragma unroll 1
            for (uint32_t j = 0; j < g; j++) {
                const uint32_t prim = ab->list[i + j]; /* warp-uniform */
                RT3_ASSERT(prim < S.n_prims);
                if (prim < S.n_faces) {
                    if (active) { exact_face<false>(S, prim, o, d, RT3_TMIN, best); }
                } else {
                    const float4 sp = __ldg(&S.spheres[prim - S.n_faces]);
                    if (active) { RT3_ABEAM_SPHERE_TEST(prim, sp, o, d, best); }
                }
            }
        }
        i += g;
    }
}

/* claim_item for the BEAM kernels: one path item per requesting lane, all from ONE chunk (so that one candidate mask
 * serves them); lanes beyond the end of the chunk go empty-handed and ask again. A new chunk gets its beam here. */
template <bool ACCEL>
__device__ __forceinline__ bool claim_item_beam(bool want, rt3_chunk& c, const rt3_kparams& P, unsigned long long* next_item, uint32_t& pixel, uint32_t& sample,
                                                const rt3_scene_view& S, const rt3_cam_view& C, rt3_beam* beam, const rt3_bvh_view& B, rt3_abeam* abeam,
                                                uint32_t* exchange, uint32_t& visits) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned m = __ballot_sync(0xffffffffu, want);
    const uint32_t n = (uint32_t) __popc(m), rank = (uint32_t) __popc(m & ((1u << lane) - 1u));
    bool got = false;
    if (n != 0u && !c.dry) {
        if (c.cur == c.end) {
            unsigned long long v = 0, size = 0;
            if (lane == 0) {
                size = chunk_size(c.start, P);
                v = atomicAdd(next_item, size);
            }
            v = __shfl_sync(0xffffffffu, v, 0);
            size = __shfl_sync(0xffffffffu, size, 0);
            if (v >= P.n_items) { c.dry = true; }
            else {
                c.cur = c.start = v;
                c.end = v + size < P.n_items ? v + size : P.n_items;
                unsigned long long p0 = v / P.spp; /* one 64-bit divide per chunk */
                c.pixel0 = (uint32_t) p0;
                c.sample0 = (uint32_t) (v - p0 * P.spp);
                if constexpr (ACCEL) { beam_for_chunk_bvh(B, C, P, c, abeam, exchange, visits); }
                else { beam_for_chunk(S, C, P, c, beam); }
            }
        }
        if (!c.dry) {
            const unsigned long long avail = c.end - c.cur;
            const uint32_t take = (unsigned long long) n < avail ? n : (uint32_t) avail;
            if (want && rank < take) {
                uint32_t k = (uint32_t) (c.cur - c.start) + rank + c.sample0; /* < spp + chunk */
                uint32_t dp = k / P.spp;
                pixel = c.pixel0 + dp;
                sample = k - dp * P.spp;
                got = true;
            }
            c.cur += (unsigned long long) take;
        }
    }
    return got;
}

/* Closest hit of a primary ray among the chunk's candidates: the exact tests in ascending primitive order with the strict
 * `t < best` rule, i.e. what the sweep's drain would report (the list is the warp's, so is the loop). */
__device__ __forceinline__ void beam_closest_hit(const rt3_scene_view& S, const rt3_beam* beam, uint32_t n_candidates, bool active, rt3_vec3 o, rt3_vec3 d, rt3_hit& best) {
    best.t = __int_as_float(0x7f800000);
    best.prim = RT3_NO_HIT;
#pragma unroll 1 /* code size: the kernel's loop has to stay inside the instruction cache */
    for (uint32_t i = 0; i < n_candidates; i++) {
        const uint32_t prim = beam->list[i];
        RT3_ASSERT(prim < S.n_prims);
        const float4 sp = __ldg(&S.spheres[prim]);
#if RT3_BEAM_EARLY_OUT
        if (active) { exact_sphere_path_coherent<true>(prim, sp, o, d, best); }
#else
        if (active) { exact_sphere_path<true>(prim, sp, o, d, best); }
#endif
    }
}

/* Persistent multi-bounce path tracer. Every thread owns RT3_RAYS path slots whose state lives in
 * shared memory; a loop iteration (1) takes the slots in turn through one copy of the shading code
 * (the hit the last sweep found), then gives every free slot of the warp the next (pixel, sample) item,
 * so that all lanes sweep live rays, and (2) sweeps the scene for all slots. */
#ifndef RT3_BEAM_CTAS_PER_SM
#define RT3_BEAM_CTAS_PER_SM 7 /* register cap 73: the BEAM kernel's regeneration would take 96 on its own; the sweep must keep its seven CTAs per SM */
#endif
#ifndef RT3_ACCEL_CTAS_PER_SM
#define RT3_ACCEL_CTAS_PER_SM 6 /* register cap 85: the traversal kernels need 77-79 and keep six CTAs per SM (without the cap ptxas drifts to 87 and five) */
#endif
template <bool RESIDENT, bool SPHERES_ONLY, bool ACCEL, int BIN = 0, bool BEAM = false>
__global__ void __launch_bounds__(RT3_CTA_THREADS, ACCEL ? RT3_ACCEL_CTAS_PER_SM : BEAM ? RT3_BEAM_CTAS_PER_SM : RT3_CTAS_PER_SM)
pathtrace_kernel(rt3_scene_view S, rt3_bvh_view B, rt3_camera cam, rt3_kparams P, unsigned long long* __restrict__ accum,
                 unsigned long long* __restrict__ counters) {
    constexpr int R = RT3_RAYS;
    static_assert(!BIN || ACCEL, "ray binning belongs to the hierarchy kernels");
    static_assert(!BEAM || (RESIDENT && (ACCEL ? (!SPHERES_ONLY && BIN != 1) : SPHERES_ONLY)),
                  "candidate lists for primary rays: resident sphere scenes through the sweep, or any scene through the hierarchy (not the CTA-wide sort)");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const rt3_smem_view sm = smem_view<RESIDENT, ACCEL>(smem_raw);
    scene_prologue<RESIDENT>(sm);
    uint32_t phase = 0u;
    rt3_bin_scratch* const bin = reinterpret_cast<rt3_bin_scratch*>(smem_raw + RT3_SLOT_BYTES); /* BIN only */
    if (BIN) { bin_prologue(B, bin); }

    rt3_cam_view C;
    C.origin = v3(cam.origin[0], cam.origin[1], cam.origin[2]);
    C.hor = v3(cam.horizontal[0], cam.horizontal[1], cam.horizontal[2]);
    C.ver = v3(cam.vertical[0], cam.vertical[1], cam.vertical[2]);
    C.llc = v3(cam.lower_left_corner[0], cam.lower_left_corner[1], cam.lower_left_corner[2]);
    C.lens_u = v3(cam.lens_u[0], cam.lens_u[1], cam.lens_u[2]);
    C.lens_v = v3(cam.lens_v[0], cam.lens_v[1], cam.lens_v[2]);
    C.lens_radius = cam.lens_radius;
    C.wm1 = (float) P.width - 1.0f; C.hm1 = (float) P.height - 1.0f;

#pragma unroll
    for (int r = 0; r < R; r++) {
#pragma unroll
        for (int fld = 0; fld < RT3_SLOT_FIELDS; fld++) { slot_word(sm, r, fld) = 0u; }
        slot_word(sm, r, RT3_F_BOUNCE) = RT3_NO_HIT;
        slot_word(sm, r, RT3_F_BEST_PRIM) = RT3_NO_HIT;
    }
    unsigned long long rays = 0;
    uint32_t visits = 0, tests = 0;
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned lane_lt = (1u << lane) - 1u;
    /* [field][this warp's 32 columns]; ACCEL + BEAM: behind the slots (and the sort scratch) */
    uint32_t* const exchange = (ACCEL ? reinterpret_cast<uint32_t*>(smem_raw + RT3_SLOT_BYTES + (BIN ? RT3_BIN_SCRATCH_BYTES : 0)) : sm.masks) + (threadIdx.x & ~31u);
    static_assert(RT3_RAYS * RT3_CHUNK_WORDS >= 8, "the exchange area needs eight mask words per thread");
    rt3_chunk chunk;
    chunk.cur = chunk.end = chunk.start = 0; chunk.pixel0 = chunk.sample0 = 0; chunk.dry = false;
    /* BEAM: this warp's candidate mask for the primary rays of its current chunk, and what went through it */
    rt3_beam* const beam = reinterpret_cast<rt3_beam*>(smem_raw + rt3_smem_bytes(RESIDENT, true)) + (threadIdx.x >> 5);
    rt3_abeam* const abeam = reinterpret_cast<rt3_abeam*>(smem_raw + RT3_SLOT_BYTES + (BIN ? RT3_BIN_SCRATCH_BYTES : 0) + RT3_ABEAM_EXCHANGE_BYTES) + (threadIdx.x >> 5); /* ACCEL */
    uint32_t beam_rays = 0, beam_tests = 0;
    chunk.beam_ok = false; chunk.beam_candidates = 0u;

    if constexpr (BEAM) {
        /* The BEAM kernel's round. One loop, one copy of the shading code: its first RT3_RAYS turns shade the slots (the hits the last
         * sweep found), the following ones are regeneration batches -- up to 32 new paths each, as many as the warp has free slots --
         * whose primary rays are traced against the candidate list of their chunk and shaded right here, in the lanes that started
         * them; what reaches a slot is the path's first BOUNCE ray (a path that ends with its primary ray never occupies one), so a
         * slot's sweeps are all spent on bounce segments. Chunks without a candidate list hand their primary rays to the slots
         * unshaded, as the other kernels do. */
        for (;;) {
            uint32_t my_rank[R];
#pragma unroll
            for (int r = 0; r < R; r++) { my_rank[r] = RT3_NO_HIT; }
            uint32_t n_free = 0, filled = 0;
#pragma unroll 1
            for (int turn = 0;; turn++) {
                const bool slot_turn = turn < R;
                /* number the warp's free slots. Wanted once, when the slot turns are over -- but a vote under a condition, even this
                 * warp-uniform one, makes ptxas give up the uniform loads of the sweep (tests/test_sass_evidence.py), so every turn votes
                 * and only turn R keeps the result */
                {
                    uint32_t rank_now[R], free_now = 0;
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        const unsigned free_r = __ballot_sync(0xffffffffu, slot_word(sm, r, RT3_F_BOUNCE) == RT3_NO_HIT);
                        rank_now[r] = ((free_r >> lane) & 1u) ? free_now + (uint32_t) __popc(free_r & lane_lt) : RT3_NO_HIT;
                        free_now += (uint32_t) __popc(free_r);
                    }
                    if (turn == R) {
                        n_free = free_now;
#pragma unroll
                        for (int r = 0; r < R; r++) { my_rank[r] = rank_now[r]; }
                    }
                }
                if (!slot_turn && (filled + (turn > R ? RT3_BEAM_MIN_BATCH : 1u) > n_free || chunk.dry || turn >= R + (int) (ACCEL ? RT3_ABEAM_BATCHES : RT3_BEAM_BATCHES))) { break; }
                rt3_path s;
                s.o = s.d = s.thr = v3(0.0f, 0.0f, 0.0f); s.key = 0u; s.pix = 0u; s.bounce = RT3_NO_HIT;
                rt3_hit best;
                best.t = __int_as_float(0x7f800000); best.prim = RT3_NO_HIT;
                bool have = false, shade = false;
                /* (votes and __syncwarp stay outside the slot-turn / batch-turn conditionals, with predicates that are false in a slot
                 * turn: under a condition they cost the sweep its uniform loads, see above) */
                const uint32_t want_n = slot_turn ? 0u : (n_free - filled < 32u ? n_free - filled : 32u);
                uint32_t p = 0, sample = 0;
                const bool got = claim_item_beam<ACCEL>(lane < want_n, chunk, P, &counters[0], p, sample, S, C, beam, B, abeam, exchange, visits);
                __syncwarp(); /* a new chunk's candidate list is in shared memory */
                if (slot_turn) {
                    s.bounce = slot_word(sm, turn, RT3_F_BOUNCE);
                    if (s.bounce != RT3_NO_HIT) {
                        s.o = slot_vec(sm, turn, RT3_F_OX); s.d = slot_vec(sm, turn, RT3_F_DX); s.thr = slot_vec(sm, turn, RT3_F_TX);
                        s.key = slot_word(sm, turn, RT3_F_KEY); s.pix = slot_word(sm, turn, RT3_F_PIX);
                        best.t = slot_float(sm, turn, RT3_F_BEST_T); best.prim = slot_word(sm, turn, RT3_F_BEST_PRIM);
                        have = shade = true;
                    }
                } else {
                    if (got) { start_path(s, C, P, p, sample); have = true; }
                    if (chunk.beam_ok) { /* warp-uniform */
                        if constexpr (ACCEL) { beam_closest_hit_bvh(S, abeam, chunk.beam_candidates, got, s.o, s.d, best); }
                        else { beam_closest_hit(S, beam, chunk.beam_candidates, got, s.o, s.d, best); }
                        shade = got;
                        if (got) { beam_rays++; beam_tests += chunk.beam_candidates; }
                    }
                }
                if (shade) { rays++; shade_path(s, best, S, P, accum); }
                const bool keep = !slot_turn && have && s.bounce != RT3_NO_HIT;
                const uint32_t keep_mask = __ballot_sync(0xffffffffu, keep);
                const uint32_t at = (uint32_t) __popc(keep_mask & lane_lt), n_made = (uint32_t) __popc(keep_mask);
                if (slot_turn) {
                    if (have) {
                        slot_word(sm, turn, RT3_F_BOUNCE) = s.bounce;
                        if (s.bounce != RT3_NO_HIT) { slot_store_vec(sm, turn, RT3_F_OX, s.o); slot_store_vec(sm, turn, RT3_F_DX, s.d); slot_store_vec(sm, turn, RT3_F_TX, s.thr); }
                    }
                } else if (keep) {
                    exchange[0 * RT3_CTA_THREADS + at] = __float_as_uint(s.o.x); exchange[1 * RT3_CTA_THREADS + at] = __float_as_uint(s.o.y);
                    exchange[2 * RT3_CTA_THREADS + at] = __float_as_uint(s.o.z); exchange[3 * RT3_CTA_THREADS + at] = __float_as_uint(s.d.x);
                    exchange[4 * RT3_CTA_THREADS + at] = __float_as_uint(s.d.y); exchange[5 * RT3_CTA_THREADS + at] = __float_as_uint(s.d.z);
                    exchange[6 * RT3_CTA_THREADS + at] = __float_as_uint(s.thr.x); exchange[7 * RT3_CTA_THREADS + at] = __float_as_uint(s.thr.y);
                    exchange[8 * RT3_CTA_THREADS + at] = __float_as_uint(s.thr.z); exchange[9 * RT3_CTA_THREADS + at] = s.key;
                    exchange[10 * RT3_CTA_THREADS + at] = s.pix; exchange[11 * RT3_CTA_THREADS + at] = s.bounce;
                }
                __syncwarp();
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const uint32_t e = my_rank[r] - filled; /* wraps around for slots that are not free, or filled already */
                    if (!slot_turn && my_rank[r] != RT3_NO_HIT && e < n_made) {
#pragma unroll
                        for (int f = 0; f < 9; f++) { slot_word(sm, r, RT3_F_OX + f) = exchange[f * RT3_CTA_THREADS + e]; }
                        slot_word(sm, r, RT3_F_KEY) = exchange[9 * RT3_CTA_THREADS + e]; slot_word(sm, r, RT3_F_PIX) = exchange[10 * RT3_CTA_THREADS + e];
                        slot_word(sm, r, RT3_F_BOUNCE) = exchange[11 * RT3_CTA_THREADS + e];
                    }
                }
                __syncwarp();
                filled += n_made;
                if (!slot_turn && !__any_sync(0xffffffffu, got)) { break; } /* the counter ran dry */
            }
            bool any = false;
#pragma unroll
            for (int r = 0; r < R; r++) { any = any || slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT; }
            if (!__any_sync(0xffffffffu, any)) {
                if (chunk.dry) { break; } /* warps run independently */
                continue;                 /* every path of this round ended with its primary ray (sky): nothing to sweep, on to the next items */
            }
            if constexpr (ACCEL) {
                if (BIN == 2) { traverse_slots_warp_sorted<false>(S, B, sm, bin, visits, tests); }
                else if (BIN == 3) { traverse_slots_warp_sorted<true>(S, B, sm, bin, visits, tests); }
                else { traverse_slots(S, B, sm, visits, tests); }
            } else {
                if (chunk.dry && warp_live_slots(sm) <= RT3_TAIL_RAYS) { sweep_slots_by_primitive(S, sm); } /* warp-uniform */
                else { sweep_slots<RESIDENT, SPHERES_ONLY>(S, sm, phase); }
            }
        }
    } else
    for (;;) {
        /* (1a) slot by slot through one copy of the shading code: shade the hit the last sweep found */
#pragma unroll 1
        for (int r = 0; r < R; r++) {
            rt3_path s;
            s.bounce = slot_word(sm, r, RT3_F_BOUNCE);
            if (s.bounce != RT3_NO_HIT) {
                s.o = slot_vec(sm, r, RT3_F_OX); s.d = slot_vec(sm, r, RT3_F_DX); s.thr = slot_vec(sm, r, RT3_F_TX);
                s.key = slot_word(sm, r, RT3_F_KEY); s.pix = slot_word(sm, r, RT3_F_PIX);
                rt3_hit best;
                best.t = slot_float(sm, r, RT3_F_BEST_T); best.prim = slot_word(sm, r, RT3_F_BEST_PRIM);
                rays++;
                shade_path(s, best, S, P, accum);
                if (!ACCEL) {
                    slot_word(sm, r, RT3_F_BOUNCE) = s.bounce;
                    if (s.bounce != RT3_NO_HIT) { slot_store_vec(sm, r, RT3_F_OX, s.o); slot_store_vec(sm, r, RT3_F_DX, s.d); slot_store_vec(sm, r, RT3_F_TX, s.thr); }
                }
            }
            if (ACCEL) {
                /* the traversal kernel regenerates slot by slot: measured 5-13 % faster there than the warp-wide form below */
                uint32_t p = 0, sample = 0;
                if (claim_item(s.bounce == RT3_NO_HIT, chunk, P, &counters[0], p, sample)) { start_path(s, C, P, p, sample); }
                slot_word(sm, r, RT3_F_BOUNCE) = s.bounce;
                if (s.bounce != RT3_NO_HIT) {
                    slot_store_vec(sm, r, RT3_F_OX, s.o); slot_store_vec(sm, r, RT3_F_DX, s.d); slot_store_vec(sm, r, RT3_F_TX, s.thr);
                    slot_word(sm, r, RT3_F_KEY) = s.key; slot_word(sm, r, RT3_F_PIX) = s.pix;
                }
            }
        }
        /* (1b) regeneration for all slots at once: the warp's free slots are numbered, and its first lanes
         * generate that many primary rays (32 per round) into an exchange area -- this warp's columns of
         * the survivor masks, which are dead between sweeps -- from where the owners of the free slots pick
         * them up. The generation code runs with as many lanes as there are free slots in the whole warp
         * instead of once per slot with a third of the lanes. */
        uint32_t my_rank[R];
        uint32_t n_free = 0;
#pragma unroll
        for (int r = 0; r < R && !ACCEL; r++) {
            const unsigned free_r = __ballot_sync(0xffffffffu, slot_word(sm, r, RT3_F_BOUNCE) == RT3_NO_HIT);
            my_rank[r] = ((free_r >> lane) & 1u) ? n_free + (uint32_t) __popc(free_r & lane_lt) : RT3_NO_HIT;
            n_free += (uint32_t) __popc(free_r);
        }
        for (uint32_t base = 0; base < n_free && !chunk.dry; base += 32u) {
            const uint32_t take = n_free - base < 32u ? n_free - base : 32u;
            rt3_path fresh;
            uint32_t p = 0, sample = 0;
            const bool got = claim_item(lane < take, chunk, P, &counters[0], p, sample);
            if (got) {
                start_path(fresh, C, P, p, sample);
                exchange[0 * RT3_CTA_THREADS + lane] = __float_as_uint(fresh.o.x); exchange[1 * RT3_CTA_THREADS + lane] = __float_as_uint(fresh.o.y);
                exchange[2 * RT3_CTA_THREADS + lane] = __float_as_uint(fresh.o.z); exchange[3 * RT3_CTA_THREADS + lane] = __float_as_uint(fresh.d.x);
                exchange[4 * RT3_CTA_THREADS + lane] = __float_as_uint(fresh.d.y); exchange[5 * RT3_CTA_THREADS + lane] = __float_as_uint(fresh.d.z);
                exchange[6 * RT3_CTA_THREADS + lane] = fresh.key; exchange[7 * RT3_CTA_THREADS + lane] = fresh.pix;
            }
            const uint32_t n_made = (uint32_t) __popc(__ballot_sync(0xffffffffu, got)); /* the claim serves the lowest lanes first */
            __syncwarp();
#pragma unroll
            for (int r = 0; r < R; r++) {
                const uint32_t e = my_rank[r] - base; /* wraps around for slots that are not free */
                if (my_rank[r] != RT3_NO_HIT && e < n_made) {
                    slot_word(sm, r, RT3_F_OX) = exchange[0 * RT3_CTA_THREADS + e]; slot_word(sm, r, RT3_F_OY) = exchange[1 * RT3_CTA_THREADS + e];
                    slot_word(sm, r, RT3_F_OZ) = exchange[2 * RT3_CTA_THREADS + e]; slot_word(sm, r, RT3_F_DX) = exchange[3 * RT3_CTA_THREADS + e];
                    slot_word(sm, r, RT3_F_DY) = exchange[4 * RT3_CTA_THREADS + e]; slot_word(sm, r, RT3_F_DZ) = exchange[5 * RT3_CTA_THREADS + e];
                    slot_word(sm, r, RT3_F_KEY) = exchange[6 * RT3_CTA_THREADS + e]; slot_word(sm, r, RT3_F_PIX) = exchange[7 * RT3_CTA_THREADS + e];
                    slot_word(sm, r, RT3_F_TX) = 0x3f800000u; slot_word(sm, r, RT3_F_TY) = 0x3f800000u; slot_word(sm, r, RT3_F_TZ) = 0x3f800000u;
                    slot_word(sm, r, RT3_F_BOUNCE) = 0u;
                }
            }
            __syncwarp();
        }
        if (BIN == 1) {
            /* the whole CTA traverses together (and leaves together) */
            if (!traverse_slots_binned(S, B, sm, bin, visits, tests)) { break; }
            continue;
        }
        bool any = false;
#pragma unroll
        for (int r = 0; r < R; r++) { any = any || slot_word(sm, r, RT3_F_BOUNCE) != RT3_NO_HIT; }
        if (RESIDENT) { if (!__any_sync(0xffffffffu, any)) { break; } }   /* warps run independently */
        else { if (!__syncthreads_or(any ? 1 : 0)) { break; } }           /* tiles are CTA-wide */
        if (BIN == 2) { traverse_slots_warp_sorted<false>(S, B, sm, bin, visits, tests); }
        else if (BIN == 3) { traverse_slots_warp_sorted<true>(S, B, sm, bin, visits, tests); }
        else if (ACCEL) { traverse_slots(S, B, sm, visits, tests); }
        else if (RESIDENT && chunk.dry && warp_live_slots(sm) <= RT3_TAIL_RAYS) { sweep_slots_by_primitive(S, sm); } /* warp-uniform */
        else { sweep_slots<RESIDENT, SPHERES_ONLY>(S, sm, phase); }
    }
    for (int off = 16; off > 0; off >>= 1) { rays += __shfl_down_sync(0xffffffffu, rays, off); }
    if ((threadIdx.x & 31) == 0 && rays) { atomicAdd(&counters[1], rays); }
    if (ACCEL) { count_accel(visits, tests, counters); }
    if (BEAM) { /* counters[2], [3] ([5], [6] in ACCEL kernels, where the hierarchy has those): primary rays traced against a candidate list, exact tests they ran */
        unsigned long long br = beam_rays, bt = beam_tests;
        for (int off = 16; off > 0; off >>= 1) { br += __shfl_down_sync(0xffffffffu, br, off); bt += __shfl_down_sync(0xffffffffu, bt, off); }
        if ((threadIdx.x & 31) == 0 && br) { atomicAdd(&counters[ACCEL ? 5 : 2], br); atomicAdd(&counters[ACCEL ? 6 : 3], bt); }
    }
}

/* ------------------------------------------------------------------------ *
 * AOVs of the path tracer's primary rays (rt3_render_path_aovs, DESIGN.md 3.7)
 * ------------------------------------------------------------------------ */

/* Signed 2^24 fixed point for the normal sums: round to nearest even, clamped to +-2^20 (as to_fixed clamps), NaN -> 0. */
__device__ __forceinline__ long long to_fixed_signed(float c) {
    float s = c * RT3_ACC_SCALE;
    if (!(s == s)) { return 0ll; }
    s = fminf(fmaxf(s, -17592186044416.0f), 17592186044416.0f); /* 2^20 * 2^24 */
    return __float2ll_rn(s);
}

/* Per-pixel sums of the AOV pass: albedo r, g, b (to_fixed), normal x, y, z (to_fixed_signed, two's complement). */
#define RT3_AOV_SUMS 6

/* One thread-ray per (pixel, sample) item, pixel-major: the primary ray start_path makes for that item, its closest hit
 * through the path tracer's tests (the path-mode sweep of the constant bank or of streamed tiles, or the hierarchy), and the
 * values shade_path sees at bounce 0 -- the albedo it multiplies by (dielectric: 1; miss: the sky of shade_miss with
 * throughput 1) and the front-facing normal (miss: 0). Item `first_sample` of a pixel also stores the pixel's primitive,
 * entity and distance along the unit direction. A warp's 32 consecutive items fall into one or two pixels once spp >= 32:
 * they are summed in the warp (a segmented scan over equal pixels) and the first lane of each pixel adds the sums with
 * six 64-bit atomics; integer sums do not depend on the order. */
template <bool RESIDENT, bool SPHERES_ONLY, bool ACCEL>
__global__ void __launch_bounds__(RT3_CTA_THREADS, RT3_REF_CTAS_PER_SM)
path_aov_kernel(rt3_scene_view S, rt3_bvh_view B, rt3_camera cam, rt3_kparams P, unsigned long long* __restrict__ sums,
                uint32_t* __restrict__ hit_prim, uint32_t* __restrict__ hit_entity, float* __restrict__ hit_t,
                unsigned long long* __restrict__ counters) {
    constexpr int R = RT3_REF_RAYS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const rt3_smem_view sm = smem_view<RESIDENT, ACCEL, RT3_MASK_BYTES_FOR(RT3_REF_RAYS)>(smem_raw);
    scene_prologue<RESIDENT>(sm);
    uint32_t phase = 0u;

    rt3_cam_view C;
    C.origin = v3(cam.origin[0], cam.origin[1], cam.origin[2]);
    C.hor = v3(cam.horizontal[0], cam.horizontal[1], cam.horizontal[2]);
    C.ver = v3(cam.vertical[0], cam.vertical[1], cam.vertical[2]);
    C.llc = v3(cam.lower_left_corner[0], cam.lower_left_corner[1], cam.lower_left_corner[2]);
    C.lens_u = v3(cam.lens_u[0], cam.lens_u[1], cam.lens_u[2]);
    C.lens_v = v3(cam.lens_v[0], cam.lens_v[1], cam.lens_v[2]);
    C.lens_radius = cam.lens_radius;
    C.wm1 = (float) P.width - 1.0f; C.hm1 = (float) P.height - 1.0f;

    rt3_vec3 o[R], d[R];
    bool live[R];
    uint32_t pixel[R], sample[R], pix[R];
    rt3_hit best[R];
    const unsigned long long cta_first = (unsigned long long) blockIdx.x * (RT3_CTA_THREADS * R);
#pragma unroll
    for (int r = 0; r < R; r++) {
        unsigned long long item = cta_first + (unsigned long long) r * RT3_CTA_THREADS + threadIdx.x;
        live[r] = item < P.n_items;
        if (!live[r]) { item = 0; }
        const unsigned long long p = item / P.spp;
        pixel[r] = (uint32_t) p; sample[r] = (uint32_t) (item - p * P.spp);
        rt3_path s;
        start_path(s, C, P, pixel[r], sample[r]);
        o[r] = s.o; d[r] = s.d; pix[r] = s.pix;
    }
    uint32_t visits = 0, tests = 0;
    if (ACCEL) {
#pragma unroll
        for (int r = 0; r < R; r++) {
            best[r].t = __int_as_float(0x7f800000); best[r].prim = RT3_NO_HIT;
            if (live[r]) { bvh_closest_hit<true>(S, B, o[r], d[r], best[r], visits, tests); }
        }
    } else {
        sweep_scene<true, RESIDENT, SPHERES_ONLY, R>(S, sm, phase, o, d, d, live, best);
    }
    const uint32_t lane = threadIdx.x & 31u;
    unsigned long long rays = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        rt3_vec3 albedo = v3(0.0f, 0.0f, 0.0f), n = v3(0.0f, 0.0f, 0.0f);
        const uint32_t prim = best[r].prim;
        if (live[r]) {
            rays++;
            if (prim == RT3_NO_HIT) {
                albedo = shade_miss(v3(1.0f, 1.0f, 1.0f), d[r], P);
            } else {
                /* shade_path's bounce-0 values, in its arithmetic */
                RT3_ASSERT(prim < S.n_prims);
                const rt3_vec3 hp = o[r] + best[r].t * d[r];
                rt3_vec3 outward;
                if (prim < S.n_faces) {
                    const float4 fn = __ldg(&S.face_rec[4 * (size_t) prim]);
                    outward = v3(fn.x, fn.y, fn.z);
                } else {
                    const float4 sp = __ldg(&S.spheres[prim - S.n_faces]);
                    const rt3_vec3 pc = hp - v3(sp.x, sp.y, sp.z);
                    outward = v3(pc.x / sp.w, pc.y / sp.w, pc.z / sp.w);
                }
                n = dot3(d[r], outward) < 0.0f ? outward : -outward;
                const uint32_t mi = __ldg(&S.prim_material[prim]);
                if (mi == RT3_NO_HIT) {
                    const float4 c = __ldg(&S.prim_color[prim]);
                    albedo = v3(c.x, c.y, c.z);
                } else {
                    const float4 m0 = __ldg(&S.materials[2 * mi]);
                    albedo = __float_as_uint(m0.x) == RT3_MAT_DIELECTRIC ? v3(1.0f, 1.0f, 1.0f) : v3(m0.y, m0.z, m0.w);
                }
            }
            if (sample[r] == 0u) {
                if (hit_prim) { hit_prim[pix[r]] = prim; }
                if (hit_entity) { hit_entity[pix[r]] = prim == RT3_NO_HIT ? RT3_NO_HIT : __ldg(&S.prim_entity[prim]); }
                if (hit_t) { hit_t[pix[r]] = best[r].t; }
            }
        }
        unsigned long long v[RT3_AOV_SUMS] = { to_fixed(albedo.x), to_fixed(albedo.y), to_fixed(albedo.z), (unsigned long long) to_fixed_signed(n.x),
                                               (unsigned long long) to_fixed_signed(n.y), (unsigned long long) to_fixed_signed(n.z) };
        /* segmented suffix scan: after it the first lane of each run of equal pixels holds the run's sums */
        const uint32_t key = live[r] ? pixel[r] : RT3_NO_HIT;
#pragma unroll
        for (uint32_t off = 1; off < 32u; off <<= 1) {
            const uint32_t other = __shfl_down_sync(0xffffffffu, key, off);
            const bool same = lane + off < 32u && other == key;
#pragma unroll
            for (int k = 0; k < RT3_AOV_SUMS; k++) {
                const unsigned long long ov = __shfl_down_sync(0xffffffffu, v[k], off);
                if (same) { v[k] += ov; }
            }
        }
        const uint32_t prev = __shfl_up_sync(0xffffffffu, key, 1);
        if (live[r] && (lane == 0u || prev != key)) {
            unsigned long long* acc = sums + RT3_AOV_SUMS * (size_t) pix[r];
#pragma unroll
            for (int k = 0; k < RT3_AOV_SUMS; k++) { if (v[k]) { atomicAdd(acc + k, v[k]); } }
        }
    }
    for (int off = 16; off > 0; off >>= 1) { rays += __shfl_down_sync(0xffffffffu, rays, off); }
    if (lane == 0 && rays) { atomicAdd(&counters[1], rays); }
    if (ACCEL) { count_accel(visits, tests, counters); }
}

/* The AOV sums as float means over the AOV samples (as radiance_kernel does for the radiance). */
__global__ void path_aov_resolve_kernel(rt3_kparams P, const unsigned long long* __restrict__ sums, float* __restrict__ albedo, float* __restrict__ normal) {
    unsigned long long p = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pixels) { return; }
    uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    size_t idx = (size_t) owned_row_to_global(P, local_row) * P.width + x;
    const double scale = (double) P.spp * (double) RT3_ACC_SCALE;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        albedo[3 * idx + c] = (float) ((double) sums[RT3_AOV_SUMS * idx + c] / scale);
        normal[3 * idx + c] = (float) ((double) (long long) sums[RT3_AOV_SUMS * idx + 3 + c] / scale);
    }
}

/* Mean over samples, gamma 2, reference packing (SequentialRenderer.cpp:297). */
__global__ void resolve_kernel(rt3_kparams P, const unsigned long long* __restrict__ accum, uint32_t* __restrict__ frame) {
    unsigned long long p = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pixels) { return; }
    uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    size_t idx = (size_t) owned_row_to_global(P, local_row) * P.width + x;
    const bool gamma = !(P.flags & RT3_FLAG_NO_GAMMA);
    uint32_t ch[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        float m = (float) ((double) accum[3 * idx + c] / ((double) P.resolve_spp * (double) RT3_ACC_SCALE));
        if (gamma) { m = sqrtf(m); }
        ch[c] = unorm8(m);
    }
    frame[idx] = (ch[0] << 24) | (ch[1] << 16) | (ch[2] << 8) | 0xFFu;
}

/* The same mean as a float image (linear radiance: before gamma and the pack), for AOV dumps. */
__global__ void radiance_kernel(rt3_kparams P, const unsigned long long* __restrict__ accum, float* __restrict__ rgb) {
    unsigned long long p = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pixels) { return; }
    uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    size_t idx = (size_t) owned_row_to_global(P, local_row) * P.width + x;
#pragma unroll
    for (int c = 0; c < 3; c++) { rgb[3 * idx + c] = (float) ((double) accum[3 * idx + c] / ((double) P.resolve_spp * (double) RT3_ACC_SCALE)); }
}

/* Clears the accumulators of the owned rows. */
__global__ void clear_accum_kernel(rt3_kparams P, unsigned long long* __restrict__ accum) {
    unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n_pixels * 3ull) { return; }
    unsigned long long p = i / 3ull;
    uint32_t c = (uint32_t) (i - p * 3ull);
    uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    size_t idx = (size_t) owned_row_to_global(P, local_row) * P.width + x;
    accum[3 * idx + c] = 0ull;
}

/* frame (full indexing) <-> compact slab of the owned rows. */
__global__ void pack_partition_kernel(rt3_kparams P, const uint32_t* __restrict__ frame, uint32_t* __restrict__ slab) {
    unsigned long long p = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pixels) { return; }
    uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    slab[p] = frame[(size_t) owned_row_to_global(P, local_row) * P.width + x];
}
__global__ void unpack_partition_kernel(rt3_kparams P, const uint32_t* __restrict__ slab, uint32_t* __restrict__ frame) {
    unsigned long long p = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pixels) { return; }
    uint32_t local_row = (uint32_t) (p / P.width), x = (uint32_t) (p - (unsigned long long) local_row * P.width);
    frame[(size_t) owned_row_to_global(P, local_row) * P.width + x] = slab[p];
}

/* Packed frame (r<<24 | g<<16 | b<<8 | a) -> interleaved 8-bit RGB or RGBA bytes, the layout image writers take
 * (reference Frame.cpp:88-96, 131-142 do this per pixel on the host). Four pixels per thread: one 16-byte
 * load, three (RGB) or four (RGBA) 4-byte stores; the tail is done per pixel. */
template <int CHANNELS>
__global__ void frame_bytes_kernel(const uint32_t* __restrict__ frame, unsigned char* __restrict__ out, unsigned long long n_pixels) {
    const unsigned long long q = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long first = 4ull * q;
    if (first >= n_pixels) { return; }
    if (first + 4ull <= n_pixels) {
        const uint4 px = *reinterpret_cast<const uint4*>(frame + first);
        /* memory order r, g, b, a = the packed word with its bytes reversed */
        const uint32_t p0 = __byte_perm(px.x, 0u, 0x0123), p1 = __byte_perm(px.y, 0u, 0x0123), p2 = __byte_perm(px.z, 0u, 0x0123),
                       p3 = __byte_perm(px.w, 0u, 0x0123);
        if (CHANNELS == 4) {
            *reinterpret_cast<uint4*>(out + 4ull * first) = make_uint4(p0 | 0xFF000000u, p1 | 0xFF000000u, p2 | 0xFF000000u, p3 | 0xFF000000u);
        } else {
            uint32_t* o = reinterpret_cast<uint32_t*>(out + 3ull * first); /* 12 bytes, 4-byte aligned because first % 4 == 0 */
            o[0] = __byte_perm(p0, p1, 0x4210); /* r0 g0 b0 r1 */
            o[1] = __byte_perm(p1, p2, 0x5421); /* g1 b1 r2 g2 */
            o[2] = __byte_perm(p2, p3, 0x6542); /* b2 r3 g3 b3 */
        }
        return;
    }
    for (unsigned long long i = first; i < n_pixels; i++) {
        const uint32_t px = frame[i];
        out[CHANNELS * i + 0] = (unsigned char) (px >> 24); out[CHANNELS * i + 1] = (unsigned char) (px >> 16); out[CHANNELS * i + 2] = (unsigned char) (px >> 8);
        if (CHANNELS == 4) { out[CHANNELS * i + 3] = 255; }
    }
}

/* FFMA throughput probe: 16 independent three-register FMA chains per thread. */
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, float a, float b, int iters) {
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; i++) { acc[i] = (float) (threadIdx.x + i); }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) { acc[i] = __fmaf_rn(acc[i], a, b); }
    }
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; i++) { s += acc[i]; }
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
