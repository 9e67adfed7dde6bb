// render.cu — the render kernels of the per-ray path (sm_100a) and their launchers.
//
// One frame = RayTracer.sample for a whole sample (ray_tracer.py:39-104): camera ray generation (camera.py:31-71),
// BVH traversal (scene.py:406-450), ray-Gaussian intersection (gaussian.py:203-230), response + SH colour
// (gaussian.py:140-201) and front-to-back compositing of the `depth` nearest entries (ray_tracer.py:79-104).
//
//   k_tile_lists + k_shade_tiles (+ k_render)   (default, RTGS_OPT_RENDER_MODE 0) the two halves of the path as separate
//                  launches: the traversal writes one candidate list per 4x8-pixel tile (tile_lists.cuh), the shading
//                  consumes them (shade.cuh), the fused kernel renders the tiles either of them handed over.  The fastest
//                  route for whole frames on one GPU (0.68 vs 0.83 ms) and for sweeps (frames on two streams overlap).
//   k_frame        (RTGS_OPT_RENDER_MODE 2) ONE launch per frame.  Persistent warps alternate between the
//                  two halves of the path: one 8x16-pixel group of the traversal (lists_group, which publishes the
//                  group's four candidate lists), then four 4x8-pixel tiles of shading (shade_tile, which acquires the
//                  publication of its tile's group).  Claims are ordered - a tile is only ever claimed after its
//                  group - so a waiting warp always waits for a warp that is running.  No kernel boundary inside the
//                  frame: the lowest LATENCY of a single frame that is spread over >= 4 GPUs (few groups per SM).
//                  Its last CTA mirrors the list-pool demand to the host.  The host queues k_render behind it for the
//                  tiles on the hand-over lists (it returns at once when they are empty); that launch completes the
//                  frame: it signals the `arrive` counter of a multi-GPU gather and zeroes the work counters for the
//                  next frame.
//   k_heavy_lists  (mode 0, opt-in RTGS_OPT_HEAVY_LISTS) depth-capped lists for the tiles of groups whose frustum overflows
//                  the traversal's shared-memory list (heavy_lists.cuh), between k_tile_lists and k_shade_tiles
//   k_render       fused.cuh (mode 1, depth > 16, fallback tiles)
//   k_generate_rays, k_trace_closest, k_activate_ply   API companions (Camera.generate_ray_field, Scene.hit, PLY ingest)
//   k_render_backward  gradient of the render with respect to the Gaussian parameters and, as
//                      k_render_backward<true> + k_camera_grad_finalize, the camera (backward.cuh)
//   k_render_rays, k_render_rays_backward   the same per-ray code for arbitrary (n,8) rays (backward.cuh)
#include <stdlib.h>

#include "backward.cuh"
#include "fused.cuh"
#include "heavy_lists.cuh"
#include "shade.cuh"
#include "tile_lists.cuh"

using namespace rtgs_dev;
using rtgs_dev::fused::k_render;

namespace {

// Release-increment at system scope: "everything before me on this stream has arrived" (bulk-copy gather).
__global__ void k_add_counter(unsigned int* counter) {
    __threadfence_system();
    asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
}

// Plain release-store at system scope (flags in mapped HOST memory, one writer each: PCIe atomics are not assumed).
__global__ void k_store_u32(unsigned int* counter, unsigned int value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(counter), "r"(value) : "memory");
}

// ---- compact delivery: float32 RGB -> float16 RGB (6 B/pixel) or RGBA8 (4 B/pixel, clipped to [0,1] and rounded
// like the reference's display path, ti.GUI.set_image, __main__.py:249-252; alpha = 255) -------------------------
__global__ void k_pack_pixels(const float* __restrict__ rgb, void* __restrict__ out, int64_t npix, int format) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (format == RTGS_PIXELS_F16) {
        // two floats -> one half2; 3 * npix floats in all (npix * 3 is even or the tail is handled singly)
        const int64_t nf = npix * 3;
        if (2 * i + 1 < nf) {
            const float2 v = *reinterpret_cast<const float2*>(rgb + 2 * i);
            reinterpret_cast<__half2*>(out)[i] = __floats2half2_rn(v.x, v.y);
        } else if (2 * i < nf) {
            reinterpret_cast<__half*>(out)[2 * i] = __float2half_rn(rgb[2 * i]);
        }
    } else if (i < npix) {
        auto q = [](float x) { return (unsigned)(fminf(fmaxf(x, 0.0f), 1.0f) * 255.0f + 0.5f); };
        const unsigned r = q(rgb[3 * i]), g = q(rgb[3 * i + 1]), b = q(rgb[3 * i + 2]);
        reinterpret_cast<unsigned*>(out)[i] = r | (g << 8) | (b << 16) | 0xff000000u;
    }
}

// ---- shared epilogue: per-warp statistics -> global counters ------------------------------------------------
template <bool STATS>
__device__ __forceinline__ void flush_lists_stats(const RenderParams& P, const ListsState& S, int lane) {
    if (STATS && P.stats && lane == 0) {
        if (S.st_nodes) atomicAdd(P.stats + ST_NODES, S.st_nodes);
        if (S.st_steps) atomicAdd(P.stats + ST_STEPS, S.st_steps);
        if (S.st_cands) atomicAdd(P.stats + ST_CANDS, S.st_cands);
        atomicMax(P.stats + ST_MAX_LISTS_STACK, (unsigned long long)S.st_max_stack);
        atomicMax(P.stats + ST_MAX_GROUP_LIST, (unsigned long long)S.st_max_list);
    }
}
template <bool STATS>
__device__ __forceinline__ void flush_shade_stats(const RenderParams& P, const ShadeStats& S, int lane) {
    if (STATS && P.stats) {
        unsigned long long v[ST_COUNT] = {0};
        v[ST_RAYS] = S.st_rays; v[ST_RAYS_HIT] = S.st_hit; v[ST_LAYERS] = S.st_layers; v[ST_F64] = S.st_f64;
        if (lane == 0) {   // warp-uniform counters are taken from lane 0 only
            v[ST_PAIRS] = 32ull * S.st_pairs;
            v[ST_TILES] = S.st_tiles;
            v[ST_INSERTS] = S.st_ins;
            v[11] = S.st_useful;
        }
#pragma unroll
        for (int k = 0; k < ST_COUNT; ++k) {
            unsigned long long x = v[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
            if (lane == 0 && x) atomicAdd(P.stats + k, x);
        }
    }
}

// ---- mode 0: the two halves as separate launches -------------------------------------------------------------
constexpr int K1_CTAS = 4;
static_assert(sizeof(ListsShared) * WARPS_PER_CTA <= 48 * 1024, "k_tile_lists: static shared-memory limit");
template <bool STATS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, K1_CTAS) k_tile_lists(const __grid_constant__ RenderParams P) {
    __shared__ ListsShared smem[WARPS_PER_CTA];
    ListsShared& ws = smem[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    ListsState S;
    const int ngroups = P.ntiles / TILES_PER_GROUP;
#pragma unroll 1
    for (;;) {
        int group = 0;
        if (lane == 0) group = (int)atomicAdd(P.counters + CTR_WORK, 1u);
        group = work_to_id(P, __shfl_sync(FULL, group, 0), P.macro_cols * GROUPS_PER_MACRO, ngroups);
        if (group >= ngroups) break;
        int gi0, gj0;
        if (!group_origin(P, group, gi0, gj0) || gi0 >= P.x0 + P.w || gj0 >= P.y0 + P.h) continue;
        lists_group<STATS>(P, ws, S, group, gi0, gj0, lane);
    }
    flush_lists_stats<STATS>(P, S, lane);
}

// ---- depth-capped lists for the tiles of the heavy groups k_tile_lists queued (heavy_lists.cuh) --------------------
constexpr int HEAVY_CTAS = 2;
template <bool STATS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, HEAVY_CTAS) k_heavy_lists(const __grid_constant__ RenderParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HeavyShared& hs = reinterpret_cast<HeavyShared*>(smem_raw)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
    ListsState S;
    HeavyStats HS;
    const int n = (int)min(P.counters[CTR_HEAVY], (unsigned)(P.ntiles / TILES_PER_GROUP)) * TILES_PER_GROUP;
    int2* def = P.heavy_scratch + ((int64_t)blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5)) * 2 * P.heavy_defer_cap;
#pragma unroll 1
    for (;;) {
        int k = 0;
        if (lane == 0) k = (int)atomicAdd(P.counters + CTR_WORK5, 1u);
        k = __shfl_sync(FULL, k, 0);
        if (k >= n) break;
        const int tile = P.heavy_groups[k / TILES_PER_GROUP] * TILES_PER_GROUP + k % TILES_PER_GROUP;
        int i0, j0;
        if (!tile_origin(P, tile, i0, j0) || i0 >= xe || j0 >= ye) continue;
        heavy_tile<STATS>(P, hs, S, HS, def, tile, i0, j0, 0.0f, lane);
        __syncwarp();
    }
    flush_lists_stats<STATS>(P, S, lane);
    if (STATS && P.stats && lane == 0) {
        if (HS.tiles) atomicAdd(P.stats + ST_HEAVY_GROUPS, HS.tiles);
        if (HS.failed) atomicAdd(P.stats + ST_HEAVY_FAILED, HS.failed);
        if (HS.iters) atomicAdd(P.stats + ST_HEAVY_PASSES, HS.iters);
        if (HS.tested) atomicAdd(P.stats + ST_HEAVY_TESTS, HS.tested);
        if (HS.retries) atomicAdd(P.stats + ST_HEAVY_RETRIES, HS.retries);
        if (HS.fail_list) atomicAdd(P.stats + ST_HEAVY_FAIL_LIST, HS.fail_list);
        if (HS.fail_defer) atomicAdd(P.stats + ST_HEAVY_FAIL_DEFER, HS.fail_defer);
        if (HS.fail_passes) atomicAdd(P.stats + ST_HEAVY_FAIL_PASSES, HS.fail_passes);
        atomicMax(P.stats + ST_MAX_DEFERRED, (unsigned long long)HS.max_deferred);
        atomicAdd(P.stats + ST_HEAVY_CYC_WALK, HS.cyc_walk);
        atomicAdd(P.stats + ST_HEAVY_CYC_TEST, HS.cyc_test);
        atomicAdd(P.stats + ST_HEAVY_CYC_PUBLISH, HS.cyc_publish);
    }
}

constexpr int K2_WARPS = 10;
constexpr int K2_CTAS = 2;
constexpr int SHADE_WARPS = K2_WARPS;   // warps per CTA
static_assert(sizeof(ShadeShared) * K2_WARPS * K2_CTAS <= 227 * 1024, "shared-memory budget per SM");

template <bool STATS, bool DEPTH = false>
__global__ void __launch_bounds__(SHADE_WARPS * 32, K2_CTAS) k_shade_tiles(const __grid_constant__ RenderParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ShadeShared& ws = reinterpret_cast<ShadeShared*>(smem_raw)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
    ShadeStats S;
    PeerGrant G;
    BandCount BC;
    grant_begin(P, G);
    band_begin(P, BC, ws.band_state, lane);
#pragma unroll 1
    for (;;) {
        int tile = 0;
        if (lane == 0) tile = (int)atomicAdd(P.counters + CTR_WORK2, 1u);
        tile = work_to_id(P, __shfl_sync(FULL, tile, 0), P.macro_cols * TILES_PER_MACRO, P.ntiles);
        if (tile >= P.ntiles) break;
        band_claim(P, BC, tile, lane);
        int i0, j0;
        if (!tile_origin(P, tile, i0, j0) || i0 >= xe || j0 >= ye) {
            tile_done(P, BC, tile, lane);
            continue;
        }
        shade_tile<STATS, DEPTH>(P, ws, S, G, BC, tile, lane);
    }
    band_flush(P, BC, lane);
    flush_shade_stats<STATS>(P, S, lane);
}

// ---- mode 2: the whole frame in one launch -------------------------------------------------------------------
union __align__(16) FrameShared {
    ListsShared lists;
    ShadeShared shade;
};
static_assert(sizeof(FrameShared) * K2_WARPS * K2_CTAS <= 227 * 1024, "shared-memory budget per SM");

template <bool STATS, bool DEPTH = false>
__global__ void __launch_bounds__(SHADE_WARPS * 32, K2_CTAS) k_frame(const __grid_constant__ RenderParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    FrameShared& ws = reinterpret_cast<FrameShared*>(smem_raw)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
    const int ngroups = P.ntiles / TILES_PER_GROUP;
    ListsState LS;
    ShadeStats SS;
    PeerGrant G;
    BandCount BC;
    grant_begin(P, G);
    band_begin(P, BC, ws.shade.band_state, lane);   // (beyond the traversal's part of the union)
    // Every warp claims ONE group, then up to FOUR tiles, and repeats.  Tile claims therefore never run ahead of
    // four times the group claims: the group of a claimed tile has been claimed by a warp that is resident and
    // does not wait for anybody, so the acquire below always terminates.  Groups and tiles run out together.
    bool groups_left = true, tiles_left = true;
#pragma unroll 1
    while (groups_left || tiles_left) {
        if (groups_left) {
            int group = 0;
            if (lane == 0) group = (int)atomicAdd(P.counters + CTR_WORK, 1u);
            group = work_to_id(P, __shfl_sync(FULL, group, 0), P.macro_cols * GROUPS_PER_MACRO, ngroups);
            int gi0, gj0;
            if (group >= ngroups) groups_left = false;
            else if (group_origin(P, group, gi0, gj0) && gi0 < xe && gj0 < ye)
                lists_group<STATS>(P, ws.lists, LS, group, gi0, gj0, lane);
        }
#pragma unroll 1
        for (int k = 0; k < TILES_PER_GROUP && tiles_left; ++k) {
            int tile = 0;
            if (lane == 0) tile = (int)atomicAdd(P.counters + CTR_WORK2, 1u);
            tile = work_to_id(P, __shfl_sync(FULL, tile, 0), P.macro_cols * TILES_PER_MACRO, P.ntiles);
            if (tile >= P.ntiles) {
                tiles_left = false;
                break;
            }
            band_claim(P, BC, tile, lane);
            int i0, j0;
            if (!tile_origin(P, tile, i0, j0) || i0 >= xe || j0 >= ye) {
                tile_done(P, BC, tile, lane);
                continue;
            }
            if (lane == 0) {   // acquire the publication of the tile's group (tile_lists.cuh)
                const unsigned int* flag = P.ready + tile / TILES_PER_GROUP;
                unsigned v;
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
                while (v != P.seq) {
                    __nanosleep(200);
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
                }
            }
            __syncwarp();
            shade_tile<STATS, DEPTH>(P, ws.shade, SS, G, BC, tile, lane);
            __syncwarp();
        }
    }
    band_flush(P, BC, lane);
    flush_lists_stats<STATS>(P, LS, lane);
    flush_shade_stats<STATS>(P, SS, lane);

    if (cta_is_last(P, CTR_DONE)) {
        // the frame's lists and shading are complete: pool demand and fallback tiles of this frame
        const unsigned pool = __ldcg(P.counters + CTR_POOL),
                       fb = __ldcg(P.counters + CTR_FALLBACK) + __ldcg(P.counters + CTR_FALLBACK2);
        *reinterpret_cast<volatile int*>(P.mirror) = (int)min(pool, 0x7fffffffu);
        if (fb != 0) *reinterpret_cast<volatile int*>(P.mirror + 1) = 1;
    }
}

// ---- multi-GPU hand-over companions (no collective on the render path: SURVEY.md 8e) -------------------------
// Wait on a stream until *counter has reached `value` (signed distance, so the 32-bit counter may wrap).
__global__ void k_wait_counter(const unsigned int* counter, unsigned int value) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    while ((int)(v - value) < 0) {
        __nanosleep(200);
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    }
}
// Raise *counter to `value` at system scope, with release semantics (everything before it on the stream is complete).
// A maximum, not a store: releases queued on different streams may execute in either order.
__global__ void k_set_counter(unsigned int* counter, unsigned int value) {
    __threadfence_system();
    asm volatile("red.release.sys.global.max.u32 [%0], %1;" ::"l"(counter), "r"(value) : "memory");
}

// ---- Camera.generate_ray_field (camera.py:57-71): (W,H,8) = origin, direction, start, end -----
__global__ void k_generate_rays(const CamD cam, float* __restrict__ rays) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= (int64_t)cam.W * cam.H) return;
    const int i = (int)(idx / cam.H), j = (int)(idx % cam.H);
    const d3 d = cam_dir(cam, (double)i + 0.5, (double)j + 0.5);
    float4* o = reinterpret_cast<float4*>(rays + idx * 8);
    o[0] = make_float4((float)cam.o[0], (float)cam.o[1], (float)cam.o[2], (float)d.x);
    o[1] = make_float4((float)d.y, (float)d.z, 0.0f, INFINITY);   // ray.py:20-41 start 0, end inf
}

// ---- Scene.hit for a batch of arbitrary rays (scene.py:406-450) -------------------------------
// Per-ray stack traversal, near child first, far-node pruning against the best entry distance.
// Box tests are float32 slabs on slightly inflated boxes; the ray-Gaussian test is the float64
// exact evaluation (this entry point exists for parity checks of closest-hit semantics, not for
// the fused renderer, which never calls it).
__global__ void k_trace_closest(const float4* __restrict__ nodes, const float4* __restrict__ raw, int64_t nrays,
                                const float* __restrict__ rays, int32_t* __restrict__ out_idx,
                                float* __restrict__ out_t12) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= nrays) return;
    const float* rp = rays + r * 8;
    const double o[3] = {rp[0], rp[1], rp[2]};
    const d3 d = d3make(rp[3], rp[4], rp[5]);
    const double t_start = rp[6], t_end = rp[7];
    const float of[3] = {rp[0], rp[1], rp[2]};
    const float idx_[3] = {1.0f / rp[3], 1.0f / rp[4], 1.0f / rp[5]};
    double best = INFINITY, best_t2 = INFINITY;
    int best_s = -1;
    int stack[RTGS_MAX_TREE_DEPTH + 2];   // depth-first, <= 2 pushes per pop: never more than depth + 1 entries
    int sp = 0;
    stack[sp++] = 0;
    auto slab = [&](float mnx, float mny, float mnz, float mxx, float mxy, float mxz) -> float {
        return slab_entry(of, idx_, {mnx, mny, mnz}, {mxx, mxy, mxz});
    };
    while (sp > 0) {
        const int node = stack[--sp];
        const float4 a = __ldg(nodes + (int64_t)node * 4 + 0), b = __ldg(nodes + (int64_t)node * 4 + 1),
                     c = __ldg(nodes + (int64_t)node * 4 + 2), dd = __ldg(nodes + (int64_t)node * 4 + 3);
        const int ch[2] = {__float_as_int(dd.x), __float_as_int(dd.y)};
        // child boxes are (centre, half extent): min = c - h, max = c + h
        float te[2] = {slab(a.x - a.w, a.y - b.x, a.z - b.y, a.x + a.w, a.y + b.x, a.z + b.y),
                       slab(b.z - c.y, b.w - c.z, c.x - c.w, b.z + c.y, b.w + c.z, c.x + c.w)};
        // visit near child first: push far first
        const int first = te[0] <= te[1] ? 0 : 1;
        for (int k = 1; k >= 0; --k) {
            const int w = k == 0 ? first : 1 - first;
            if (!(te[w] < INFINITY) || (double)te[w] > best) continue;   // miss or farther than best
            if (ch[w] >= 0) {
                stack[sp++] = ch[w];
            } else {
                const int s = ~ch[w];
                const float4 ra = __ldg(raw + (int64_t)s * 3 + 0), rb = __ldg(raw + (int64_t)s * 3 + 1),
                             rc = __ldg(raw + (int64_t)s * 3 + 2);
                const double p[3] = {ra.x, ra.y, ra.z}, q[4] = {ra.w, rb.x, rb.y, rb.z}, sc[3] = {rb.w, rc.x, rc.y};
                const ExactHit e = exact_intersect(p, q, sc, o, d);
                if (e.hit && e.t1 > t_start && e.t1 < t_end && e.t1 < best) {   // scene.py:433-437
                    best = e.t1;
                    best_t2 = e.t2;
                    best_s = s;
                }
            }
        }
    }
    if (best_s >= 0) {
        out_idx[r] = __float_as_int(__ldg(raw + (int64_t)best_s * 3 + 2).z);
        out_t12[r * 2 + 0] = (float)best;
        out_t12[r * 2 + 1] = (float)best_t2;
    } else {
        out_idx[r] = -1;
        out_t12[r * 2 + 0] = INFINITY;
        out_t12[r * 2 + 1] = INFINITY;
    }
}

// ---- PLY rows -> stored parameters (scene.py:101-114 on the device) ---------------------------
__global__ void k_activate_ply(int64_t n, const float* __restrict__ rows, int stride, const int32_t* __restrict__ col,
                               float scale_arg, int sh_layout, float* __restrict__ pos, float* __restrict__ rot,
                               float* __restrict__ sca, float* __restrict__ color, float* __restrict__ opacity,
                               float* __restrict__ sh) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* row = rows + i * stride;
    auto get = [&](int k) -> float { int c = col[k]; return c >= 0 ? row[c] : 0.0f; };
    // column order: x,y,z (0-2), f_dc (3-5), f_rest (6-50), opacity (51), scale (52-54), rot_0..3 (55-58)
    pos[i * 3 + 0] = get(0); pos[i * 3 + 1] = get(1); pos[i * 3 + 2] = get(2);
    // scalar-first (rot_0 = w) -> scalar-last, normalised in float32 (scene.py:103,110-111)
    const float qx = get(56), qy = get(57), qz = get(58), qw = get(55);
    const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(qx, qx), __fmul_rn(qy, qy)), __fmul_rn(qz, qz)),
                                           __fmul_rn(qw, qw)));
    rot[i * 4 + 0] = __fdiv_rn(qx, nrm); rot[i * 4 + 1] = __fdiv_rn(qy, nrm);
    rot[i * 4 + 2] = __fdiv_rn(qz, nrm); rot[i * 4 + 3] = __fdiv_rn(qw, nrm);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        sca[i * 3 + a] = __fmul_rn(expf(get(52 + a)), scale_arg);                  // scene.py:112
        color[i * 3 + a] = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-get(3 + a))));     // scene.py:113
    }
    opacity[i] = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-get(51))));                 // scene.py:114
    if (sh != nullptr) {
        for (int k = 0; k < 15; ++k)
            for (int c = 0; c < 3; ++c)
                sh[i * 45 + k * 3 + c] = sh_layout == 0 ? get(6 + 15 * c + k) : get(6 + 3 * k + c);
    }
}

CamD make_camd(const rtgs_camera* cam) {
    CamD c;
    for (int a = 0; a < 3; ++a) c.o[a] = cam->position[a];
    for (int a = 0; a < 4; ++a) c.q[a] = cam->rotation[a];
    double Rm[3][3];
    quat_to_mat(c.q, Rm);   // utils/quaternion.py:99-121 in float64 (rotation used as given, not normalised)
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) c.R[r * 3 + k] = Rm[r][k];
    c.fx = cam->focal[0];
    c.fy = cam->focal[1];
    c.ifx = 1.0 / c.fx;
    c.ify = 1.0 / c.fy;
    c.W = cam->width;
    c.H = cam->height;
    return c;
}

int device_slot(const rtgs_scene* s) { return s->device >= 0 && s->device < 16 ? s->device : 0; }

// Occupancy of a persistent kernel on the scene's device (cached per device), with its dynamic shared memory opted in.
template <typename Kernel>
int persistent_blocks(rtgs_scene* s, Kernel kernel, int threads, size_t smem, int* cache, const char* name, int* out) {
    const int dev = device_slot(s);
    if (cache[dev] == 0) {
        if (smem > 0) CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int nb = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem));
        if (nb < 1) {
            rtgs_set_error("%s does not fit on an SM (smem %zu)", name, smem);
            return RTGS_ERR_CUDA;
        }
        cache[dev] = nb;
    }
    *out = cache[dev];
    return RTGS_OK;
}

template <int K, bool STATS, bool DEPTH>
int launch_render_k(rtgs_scene* s, const rtgs_scene::FrameScratch& fs, const RenderParams& P, cudaStream_t stream) {
    static int cache[16] = {0};
    const size_t smem = sizeof(fused::WarpShared<K>) * WARPS_PER_CTA;
    int nb = 0;
    int r = persistent_blocks(s, k_render<K, STATS, DEPTH>, WARPS_PER_CTA * 32, smem, cache, "k_render", &nb);
    if (r != RTGS_OK) return r;
    int grid = s->sm_count * nb;
    const int need = (P.ntiles + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    if (grid > need) grid = need;
    if (P.use_fallback_list) {
        // The fallback launch is empty unless the list pool overflowed.  While no finished frame has reported
        // fallback tiles it runs on a quarter of the SMs (a cheaper launch); the first frame that does overflow
        // is still rendered correctly, just with fewer warps on its fallback tiles.
        const int seen = *reinterpret_cast<volatile int*>(fs.mirror + 1);
        const int small = (s->sm_count + 3) / 4;
        if (!seen && grid > small) grid = small;
    }
    if (grid < 1) grid = 1;
    k_render<K, STATS, DEPTH><<<grid, WARPS_PER_CTA * 32, smem, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

template <bool STATS, bool DEPTH>
int launch_fused(rtgs_scene* s, const rtgs_scene::FrameScratch& fs, const RenderParams& P, cudaStream_t stream, int K) {
    return K > 16 ? launch_render_k<32, STATS, DEPTH>(s, fs, P, stream) : launch_render_k<16, STATS, DEPTH>(s, fs, P, stream);
}

template <bool STATS>
int launch_tile_lists(rtgs_scene* s, const RenderParams& P, cudaStream_t stream) {
    static int cache[16] = {0};
    int nb = 0;
    int r = persistent_blocks(s, k_tile_lists<STATS>, WARPS_PER_CTA * 32, 0, cache, "k_tile_lists", &nb);
    if (r != RTGS_OK) return r;
    int grid = s->sm_count * nb;
    const int need = (P.ntiles / TILES_PER_GROUP + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    k_tile_lists<STATS><<<grid, WARPS_PER_CTA * 32, 0, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

// Deferred-node lists of k_heavy_lists: two of HEAVY_DEFER_CAP entries per warp of its grid (allocated on first use).
constexpr int HEAVY_DEFER_CAP = 2048;
template <bool STATS>
int launch_heavy_lists(rtgs_scene* s, rtgs_scene::FrameScratch& fs, RenderParams& P, cudaStream_t stream) {
    static int cache[16] = {0};
    const size_t smem = sizeof(HeavyShared) * WARPS_PER_CTA;
    int nb = 0;
    int r = persistent_blocks(s, k_heavy_lists<STATS>, WARPS_PER_CTA * 32, smem, cache, "k_heavy_lists", &nb);
    if (r != RTGS_OK) return r;
    if (nb > HEAVY_CTAS) nb = HEAVY_CTAS;
    int grid = s->sm_count * nb;
    const int need = (P.ntiles + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    const int warps = grid * WARPS_PER_CTA;
    if (fs.heavy_scratch_warps < warps) {
        cudaFree(fs.heavy_scratch);
        fs.heavy_scratch = nullptr;
        fs.heavy_scratch_warps = 0;
        CUDA_TRY(cudaMalloc((void**)&fs.heavy_scratch, (size_t)warps * 2 * HEAVY_DEFER_CAP * sizeof(int2)));
        fs.heavy_scratch_warps = warps;
    }
    P.heavy_scratch = fs.heavy_scratch;
    P.heavy_defer_cap = HEAVY_DEFER_CAP;
    k_heavy_lists<STATS><<<grid, WARPS_PER_CTA * 32, smem, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

template <bool STATS, bool DEPTH>
int launch_shade_tiles(rtgs_scene* s, const RenderParams& P, cudaStream_t stream) {
    static int cache[16] = {0};
    const size_t smem = sizeof(ShadeShared) * SHADE_WARPS;
    int nb = 0;
    int r = persistent_blocks(s, k_shade_tiles<STATS, DEPTH>, SHADE_WARPS * 32, smem, cache, "k_shade_tiles", &nb);
    if (r != RTGS_OK) return r;
    int grid = s->sm_count * nb;
    const int need = (P.ntiles + SHADE_WARPS - 1) / SHADE_WARPS;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    k_shade_tiles<STATS, DEPTH><<<grid, SHADE_WARPS * 32, smem, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

template <bool STATS, bool DEPTH>
int launch_frame(rtgs_scene* s, const RenderParams& P, cudaStream_t stream) {
    static int cache[16] = {0};
    const size_t smem = sizeof(FrameShared) * SHADE_WARPS;
    int nb = 0;
    int r = persistent_blocks(s, k_frame<STATS, DEPTH>, SHADE_WARPS * 32, smem, cache, "k_frame", &nb);
    if (r != RTGS_OK) return r;
    int grid = s->sm_count * nb;
    // a warp does one group and four tiles per round: more warps than groups would only spin
    const int need = (P.ntiles / TILES_PER_GROUP + SHADE_WARPS - 1) / SHADE_WARPS;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    k_frame<STATS, DEPTH><<<grid, SHADE_WARPS * 32, smem, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

// Which kernels render a frame: 0 (default) = k_tile_lists + k_shade_tiles + k_render on the fallback list; 2 =
// k_frame, one launch (lowest latency of a single frame that is spread over >= 4 GPUs); 1 = the fused k_render
// alone.  depth > 16 always takes the fused kernel (32-entry k-buffer).
int render_mode(const rtgs_scene* s) {
    if (s->opt_render_mode >= 0) return s->opt_render_mode;
    static int mode = -1;
    if (mode < 0) {
        const char* e = getenv("RTGS_RENDER_MODE");
        mode = e ? atoi(e) : 0;
        if (mode < 0 || mode > 2) mode = 0;
    }
    return mode;
}

}  // namespace

// Heavy groups (heavy_lists.cuh): 0 (default) = the fused kernel renders their tiles, 1 = depth-capped lists once the
// scene has shown heavy groups, 2 = from the first frame on.  Off by default: on the surface-like scene the two routes
// cost the same (DESIGN.md §8), and the fused kernel is the simpler one.
int rtgs_heavy_lists_mode(const rtgs_scene* s) { return s->opt_heavy_lists >= 0 ? s->opt_heavy_lists : 0; }

namespace {
// Candidate-list scratch of a scene, sized for the tile count of the largest region rendered so far.
// The pool starts at 16 chunks (496 candidates) per tile on average - tiles may take any share of it - and
// doubles whenever the demand reported by the last finished frame (lists_group keeps counting past the end of
// the pool; the frame's last CTA mirrors the count into mapped host memory) exceeded 70 % of it.  A frame
// that overflows is still rendered correctly (fallback list), the next one has the larger pool.
int ensure_lists(rtgs_scene* s, rtgs_scene::FrameScratch& fs, int ntiles) {
    int64_t want = fs.pool_chunks;
    if (s->opt_pool_chunks < 0 && fs.list_tiles > 0) {
        const int64_t used = *reinterpret_cast<volatile int*>(fs.mirror);
        while (used * 10 > want * 7 && want < (1ll << 26)) want *= 2;
    }
    if (fs.list_tiles >= ntiles && want == fs.pool_chunks) return RTGS_OK;
    const bool grow_only = fs.list_tiles >= ntiles;
    const int tiles = grow_only ? fs.list_tiles : ntiles;
    cudaFree(fs.tile_desc); cudaFree(fs.list_pool); cudaFree(fs.fallback_tiles); cudaFree(fs.fallback_tiles2); cudaFree(fs.ready);
    cudaFree(fs.heavy_groups); cudaFree(fs.tile_cap);
    fs.tile_desc = nullptr; fs.list_pool = nullptr; fs.fallback_tiles = nullptr; fs.fallback_tiles2 = nullptr; fs.ready = nullptr;
    fs.heavy_groups = nullptr; fs.tile_cap = nullptr;
    fs.list_tiles = 0;
    int64_t chunks = s->opt_pool_chunks >= 0 ? s->opt_pool_chunks : (int64_t)tiles * 16;
    if (grow_only && want > chunks) chunks = want;
    if (chunks > (1ll << 26)) chunks = 1ll << 26;
    CUDA_TRY(cudaMalloc((void**)&fs.tile_desc, (size_t)tiles * sizeof(TileDesc)));
    CUDA_TRY(cudaMalloc((void**)&fs.list_pool, (size_t)(chunks > 0 ? chunks : 1) * CHUNK_INTS * sizeof(int)));
    CUDA_TRY(cudaMalloc((void**)&fs.fallback_tiles, (size_t)tiles * sizeof(int)));
    CUDA_TRY(cudaMalloc((void**)&fs.fallback_tiles2, (size_t)tiles * sizeof(int)));
    CUDA_TRY(cudaMalloc((void**)&fs.heavy_groups, ((size_t)tiles / TILES_PER_GROUP + 1) * sizeof(int)));
    CUDA_TRY(cudaMalloc((void**)&fs.tile_cap, (size_t)tiles * sizeof(float)));
    // group publication flags: compared with the frame sequence number, which starts at 1 and never repeats
    const size_t groups = (size_t)tiles / TILES_PER_GROUP + 1;
    CUDA_TRY(cudaMalloc((void**)&fs.ready, groups * sizeof(unsigned int)));
    CUDA_TRY(cudaMemset(fs.ready, 0, groups * sizeof(unsigned int)));
    fs.list_tiles = tiles;
    fs.pool_chunks = (int)chunks;
    fs.mirror[0] = 0;
    return RTGS_OK;
}

}  // namespace

static int launch_render_on(rtgs_scene* s, rtgs_scene::FrameScratch& fs, const rtgs_camera* cam, int x0, int y0, int w,
                            int h, int depth, float t_cut, int accumulate, int full_pitch, float* out_rgb,
                            float* out_T, float* out_depth, cudaStream_t stream, bool want_stats);

// A frame's render scratch (work counters, candidate lists) is reused by later frames, which is safe in stream
// order.  The scene has two scratch sets: a stream keeps the set it used last, a new stream takes the set that has
// been idle longest and first waits for that set's last frame.  So frames launched alternately on two streams never
// wait for each other and overlap on the device; a third stream, or statistics / banded delivery (whose counters
// exist once), are ordered behind what they share.
int rtgs_launch_render(rtgs_scene* s, const rtgs_camera* cam, int x0, int y0, int w, int h, int depth,
                       float t_cut, int accumulate, int full_pitch, float* out_rgb, float* out_T, float* out_depth,
                       cudaStream_t stream, bool want_stats) {
    const bool exclusive = want_stats || s->bands_active > 0;   // uses stats_dev / band_done: one frame at a time
    int pick = -1;
    for (int k = 0; k < 2; ++k)
        if (s->scratch[k].used && s->scratch[k].stream == stream) pick = k;
    if (pick < 0) pick = (!s->scratch[0].used || (s->scratch[1].used && s->scratch[0].last_use < s->scratch[1].last_use)) ? 0 : 1;
    if (exclusive) pick = 0;
    rtgs_scene::FrameScratch& fs = s->scratch[pick];
    for (int k = 0; k < 2; ++k) {
        rtgs_scene::FrameScratch& o = s->scratch[k];
        if (o.used && o.stream != stream && (k == pick || exclusive || s->exclusive_inflight))
            CUDA_TRY(cudaStreamWaitEvent(stream, o.free_event, 0));
    }
    s->exclusive_inflight = exclusive;
    const int r = launch_render_on(s, fs, cam, x0, y0, w, h, depth, t_cut, accumulate, full_pitch, out_rgb, out_T,
                                   out_depth, stream, want_stats);
    // the hand-over pointers apply to one frame
    s->sync_arrive = nullptr;
    s->sync_grant = nullptr;
    // (also after a failed launch sequence: whatever was queued still uses the scratch)
    if (cudaEventRecord(fs.free_event, stream) == cudaSuccess) {
        fs.stream = stream;
        fs.used = true;
        fs.last_use = ++s->scratch_clock;
    } else {
        cudaGetLastError();
    }
    return r;
}

static int launch_render_on(rtgs_scene* s, rtgs_scene::FrameScratch& fs, const rtgs_camera* cam, int x0, int y0, int w,
                            int h, int depth, float t_cut, int accumulate, int full_pitch, float* out_rgb,
                            float* out_T, float* out_depth, cudaStream_t stream, bool want_stats) {
    RenderParams P;
    P.nodes = s->nodes;
    P.nodes4 = s->nodes4;
    P.geo = s->geo;
    P.shp = s->shp;
    P.shp_tex = s->shp_tex;
    P.raw = s->raw;
    P.leafbox = s->leafbox;
    P.cam = make_camd(cam);
    P.x0 = x0; P.y0 = y0; P.w = w; P.h = h;
    const int mrows = (w + MACRO_PX_I - 1) / MACRO_PX_I;
    const int mcols = (h + MACRO_PX_J - 1) / MACRO_PX_J;
    P.macro_cols = mcols;
    P.stripe_mod = s->opt_stripe_mod;
    P.stripe_rem = s->opt_stripe_rem;
    P.ntiles = mrows * mcols * TILES_PER_MACRO;
    P.depth = depth;
    P.t_cut = t_cut;
    P.accumulate = accumulate;
    P.full_pitch = full_pitch;
    P.has_sh = s->has_sh ? 1 : 0;
    P.out_rgb = out_rgb;
    P.out_T = out_T;
    P.counters = fs.counters;
    P.stats = want_stats ? s->stats_dev : nullptr;
    P.desc = nullptr;
    P.pool = nullptr;
    P.pool_chunks = 0;
    P.fallback_tiles = nullptr;
    P.fallback_tiles2 = nullptr;
    P.use_fallback_list = 0;
    static const int heavy_fused = getenv("RTGS_HEAVY_FUSED") ? atoi(getenv("RTGS_HEAVY_FUSED")) : 1;
    P.heavy_fused = heavy_fused;
    P.heavy_limit = s->opt_heavy_limit >= 0 ? s->opt_heavy_limit : 1 << 30;   // default: the shared list's capacity
    P.heavy_slab = 0;
    P.heavy_groups = nullptr;
    P.tile_cap = nullptr;
    P.heavy_scratch = nullptr;
    P.heavy_defer_cap = 0;
    // batch threshold of the traversal stack: the tuned value, capped by what this tree's depth allows (>= 4)
    P.lists_single = min(LISTS_SINGLE, lists_single_bound(s->max_depth));
    P.nbands = 0;
    P.band_macro_cols = 1;
    P.macro_rows = mrows;
    P.schedule = s->bands_active > 0 ? 2 : 0;
    P.band_done = s->band_done;
    P.band_flags = s->band_flags_cur_dev ? s->band_flags_cur_dev : s->band_flags_dev;
    P.mirror = fs.mirror_dev;
    P.ready = nullptr;
    P.seq = 0;
    P.arrive = s->sync_arrive;
    P.grant = s->sync_grant;
    P.grant_value = s->sync_grant_value;
    P.final_kernel = 0;
    P.self_clean = 0;
    P.out_depth = out_depth;
    // out_depth selects the DEPTH instantiation of every kernel that composites; without it the frame runs the kernels
    // of a plain render
    const bool with_depth = out_depth != nullptr;
    if (s->bands_active > 0) {
        P.nbands = s->bands_active;
        P.band_macro_cols = s->band_macro_cols;
        CUDA_TRY(cudaMemsetAsync(s->band_done, 0, RTGS_MAX_BANDS * sizeof(unsigned int), stream));
    }
    const int mode = depth > 16 ? 1 : render_mode(s);
    // work counters: k_frame's last CTA leaves them zeroed for the next frame; the other modes (and the first
    // frame after one of them) reset them here
    const bool self_clean = mode == 2;
    if (!self_clean || fs.counters_dirty) CUDA_TRY(cudaMemsetAsync(fs.counters, 0, CTR_COUNT * sizeof(unsigned int), stream));
    fs.counters_dirty = !self_clean;
    if (want_stats) CUDA_TRY(cudaMemsetAsync(s->stats_dev, 0, ST_TOTAL * sizeof(unsigned long long), stream));

    // optional per-kernel timing: events e[0..3] of this frame's ring slot bracket up to three launches
    cudaEvent_t* ev = nullptr;
    unsigned char* ran = nullptr;
    if (!s->timing_ran.empty()) {
        const int64_t slot = s->timing_frames % (int64_t)s->timing_ran.size();
        ev = &s->timing_events[slot * 4];
        ran = &s->timing_ran[slot];
        *ran = 0;
        ++s->timing_frames;
    }
    auto mark = [&](int k) -> int {
        if (ev) CUDA_TRY(cudaEventRecord(ev[k], stream));
        return RTGS_OK;
    };
    // f<STATS, DEPTH>(...) for this frame's statistics and depth flags
#define RTGS_BY_FLAGS(f, ...)                                                                                         \
    (want_stats ? (with_depth ? f<true, true>(__VA_ARGS__) : f<true, false>(__VA_ARGS__))                               \
                : (with_depth ? f<false, true>(__VA_ARGS__) : f<false, false>(__VA_ARGS__)))
    auto fused_kernel = [&](int K) -> int { return RTGS_BY_FLAGS(launch_fused, s, fs, P, stream, K); };
    int r;
    if (mode == 1) {
        if ((r = mark(0)) != RTGS_OK || (r = mark(1)) != RTGS_OK || (r = mark(2)) != RTGS_OK) return r;
        P.final_kernel = 1;
        if ((r = fused_kernel(depth > 16 ? 32 : 16)) != RTGS_OK) return r;
        if (ran) *ran = 4;
        return mark(3);
    }
    // traversal -> per-tile candidate lists -> shading; tiles whose list did not fit the pool (or whose group holds
    // too many candidates) are rendered by the fused kernel behind them
    if ((r = ensure_lists(s, fs, P.ntiles)) != RTGS_OK) return r;
    P.desc = reinterpret_cast<TileDesc*>(fs.tile_desc);
    P.pool = fs.list_pool;
    P.pool_chunks = fs.pool_chunks;
    P.fallback_tiles = fs.fallback_tiles;
    P.fallback_tiles2 = fs.fallback_tiles2;
    if (mode == 2) {
        P.ready = fs.ready;
        P.seq = ++fs.frame_seq;
        if ((r = mark(0)) != RTGS_OK || (r = mark(1)) != RTGS_OK) return r;
        if ((r = RTGS_BY_FLAGS(launch_frame, s, P, stream)) != RTGS_OK) return r;
        if ((r = mark(2)) != RTGS_OK) return r;
        P.use_fallback_list = 1;
        P.final_kernel = 1;
        P.self_clean = 1;
        if ((r = fused_kernel(16)) != RTGS_OK) return r;
        if (ran) *ran = 6;
        return mark(3);
    }
    // Groups whose frustum overflows the traversal's shared-memory list ("heavy") go to the fused kernel.  With
    // RTGS_OPT_HEAVY_LISTS = 1 (2) the traversal queues them instead, once a frame of this scene has reported some
    // (from the first frame on), and k_heavy_lists lists their tiles in depth slabs (heavy_lists.cuh); scenes without
    // heavy groups never launch the extra kernel.  (Its time is counted with k_tile_lists.)
    P.tile_cap = fs.tile_cap;
    P.heavy_groups = fs.heavy_groups;
    const int heavy_mode = rtgs_heavy_lists_mode(s);
    const bool heavy_seen = *reinterpret_cast<volatile int*>(s->scratch[0].mirror + 2) != 0 ||
                            *reinterpret_cast<volatile int*>(s->scratch[1].mirror + 2) != 0;
    P.heavy_slab = (heavy_mode == 2 || (heavy_mode == 1 && heavy_seen)) ? 1 : 0;
    if ((r = mark(0)) != RTGS_OK) return r;
    if ((r = want_stats ? launch_tile_lists<true>(s, P, stream) : launch_tile_lists<false>(s, P, stream)) != RTGS_OK) return r;
    if (P.heavy_slab &&
        (r = want_stats ? launch_heavy_lists<true>(s, fs, P, stream) : launch_heavy_lists<false>(s, fs, P, stream)) != RTGS_OK)
        return r;
    if ((r = mark(1)) != RTGS_OK) return r;
    if ((r = RTGS_BY_FLAGS(launch_shade_tiles, s, P, stream)) != RTGS_OK) return r;
    if ((r = mark(2)) != RTGS_OK) return r;
    // the closing launch renders both hand-over lists
    P.use_fallback_list = 1;
    P.final_kernel = 1;
    if ((r = fused_kernel(16)) != RTGS_OK) return r;
    if (ran) *ran = 7;
    return mark(3);
#undef RTGS_BY_FLAGS
}

int rtgs_launch_generate_rays(const rtgs_camera* cam, float* rays, cudaStream_t stream) {
    const CamD c = make_camd(cam);
    const int64_t n = (int64_t)c.W * c.H;
    k_generate_rays<<<(int)((n + 255) / 256), 256, 0, stream>>>(c, rays);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_trace_closest(rtgs_scene* s, int64_t nrays, const float* rays, int32_t* idx, float* t12,
                              cudaStream_t stream) {
    if (nrays == 0) return RTGS_OK;
    k_trace_closest<<<(int)((nrays + 127) / 128), 128, 0, stream>>>(s->nodes, s->raw, nrays, rays, idx, t12);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_render_backward(rtgs_scene* s, const rtgs_camera* cam, int x0, int y0, int w, int h, int depth,
                                float t_cut, const float* dL_drgb, const float* dL_dT, const float* dL_dD,
                                float* const grads[6], float* const cam_grads[3], float* replay_rgb, float* replay_T,
                                float* replay_depth, cudaStream_t stream) {
    backward::BackwardParams P;
    P.nodes = s->nodes;
    P.geo = s->geo;
    P.shp = s->shp;
    P.raw = s->raw;
    P.cam = make_camd(cam);
    P.x0 = x0; P.y0 = y0; P.w = w; P.h = h;
    P.tiles_j = (h + TILE_J - 1) / TILE_J;
    P.ntiles = ((w + TILE_I - 1) / TILE_I) * P.tiles_j;
    P.depth = depth;
    P.t_cut = t_cut;
    P.has_sh = s->has_sh ? 1 : 0;
    P.dL_drgb = dL_drgb;
    P.dL_dT = dL_dT;
    P.g_pos = grads[0]; P.g_rot = grads[1]; P.g_scale = grads[2];
    P.g_color = grads[3]; P.g_opacity = grads[4]; P.g_sh = s->has_sh ? grads[5] : nullptr;
    P.replay_rgb = replay_rgb;
    P.replay_T = replay_T;
    P.dL_dD = dL_dD;
    P.replay_depth = replay_depth;
    P.cam_part = nullptr;
    // the DEPTH instantiations only when a depth pointer is given: otherwise the kernels of the plain backward
    const bool with_depth = dL_dD != nullptr || replay_depth != nullptr;
    const int blocks = (P.ntiles + backward::BWD_WARPS - 1) / backward::BWD_WARPS;
    if (cam_grads[0] == nullptr && cam_grads[1] == nullptr && cam_grads[2] == nullptr) {
        if (with_depth) backward::k_render_backward<false, true><<<blocks, backward::BWD_WARPS * 32, 0, stream>>>(P);
        else backward::k_render_backward<false><<<blocks, backward::BWD_WARPS * 32, 0, stream>>>(P);
        CUDA_TRY(cudaGetLastError());
        return RTGS_OK;
    }
    // per-CTA partials of the camera gradient, stream-ordered: no scene scratch, safe for calls on several streams
    CUDA_TRY(cudaMallocAsync((void**)&P.cam_part, sizeof(double) * backward::CAM_TERMS * blocks, stream));
    if (with_depth) backward::k_render_backward<true, true><<<blocks, backward::BWD_WARPS * 32, 0, stream>>>(P);
    else backward::k_render_backward<true><<<blocks, backward::BWD_WARPS * 32, 0, stream>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) {
        backward::k_camera_grad_finalize<<<1, backward::FIN_THREADS, 0, stream>>>(P.cam_part, blocks, P.cam, cam_grads[0],
                                                                                   cam_grads[1], cam_grads[2]);
        e = cudaGetLastError();
    }
    const cudaError_t ef = cudaFreeAsync(P.cam_part, stream);
    CUDA_TRY(e);
    CUDA_TRY(ef);
    return RTGS_OK;
}

// The parameters of the ray kernels (no camera, no region); dL, gradient and output pointers are set by the caller.
static backward::BackwardParams rays_params(rtgs_scene* s, int64_t nrays, const float* rays, int depth, float t_cut) {
    backward::BackwardParams P = {};
    P.nodes = s->nodes;
    P.geo = s->geo;
    P.shp = s->shp;
    P.raw = s->raw;
    P.depth = depth;
    P.t_cut = t_cut;
    P.has_sh = s->has_sh ? 1 : 0;
    P.rays = rays;
    P.nrays = nrays;
    return P;
}

int rtgs_launch_render_rays(rtgs_scene* s, int64_t nrays, const float* rays, int depth, float t_cut, float* out_rgb,
                            float* out_T, float* out_depth, cudaStream_t stream) {
    if (nrays == 0) return RTGS_OK;
    backward::BackwardParams P = rays_params(s, nrays, rays, depth, t_cut);
    P.replay_rgb = out_rgb;
    P.replay_T = out_T;
    P.replay_depth = out_depth;
    const unsigned blocks = (unsigned)((nrays + backward::RAY_THREADS - 1) / backward::RAY_THREADS);
    if (out_depth != nullptr) backward::k_render_rays<true><<<blocks, backward::RAY_THREADS, 0, stream>>>(P);
    else backward::k_render_rays<<<blocks, backward::RAY_THREADS, 0, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_render_rays_backward(rtgs_scene* s, int64_t nrays, const float* rays, int depth, float t_cut,
                                     const float* dL_drgb, const float* dL_dT, const float* dL_dD,
                                     float* const grads[6], float* grad_rays, float* replay_rgb, float* replay_T,
                                     float* replay_depth, cudaStream_t stream) {
    if (nrays == 0) return RTGS_OK;
    backward::BackwardParams P = rays_params(s, nrays, rays, depth, t_cut);
    P.dL_drgb = dL_drgb;
    P.dL_dT = dL_dT;
    P.g_pos = grads[0]; P.g_rot = grads[1]; P.g_scale = grads[2];
    P.g_color = grads[3]; P.g_opacity = grads[4]; P.g_sh = s->has_sh ? grads[5] : nullptr;
    P.g_rays = grad_rays;
    P.replay_rgb = replay_rgb;
    P.replay_T = replay_T;
    P.dL_dD = dL_dD;
    P.replay_depth = replay_depth;
    const unsigned blocks = (unsigned)((nrays + backward::RAY_THREADS - 1) / backward::RAY_THREADS);
    const bool with_depth = dL_dD != nullptr || replay_depth != nullptr;
    if (grad_rays == nullptr && !with_depth)
        backward::k_render_rays_backward<false><<<blocks, backward::RAY_THREADS, 0, stream>>>(P);
    else if (grad_rays == nullptr)
        backward::k_render_rays_backward<false, true><<<blocks, backward::RAY_THREADS, 0, stream>>>(P);
    else if (!with_depth)
        backward::k_render_rays_backward<true><<<blocks, backward::RAY_THREADS, 0, stream>>>(P);
    else
        backward::k_render_rays_backward<true, true><<<blocks, backward::RAY_THREADS, 0, stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_activate_ply(int64_t n, const float* rows_dev, int stride, const int32_t* col, float scale,
                             int sh_layout, float* pos, float* rot, float* sca, float* color, float* opacity,
                             float* sh, cudaStream_t stream) {
    k_activate_ply<<<(int)((n + 127) / 128), 128, 0, stream>>>(n, rows_dev, stride, col, scale, sh_layout, pos, rot,
                                                               sca, color, opacity, sh);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_wait_counter(const unsigned int* counter, unsigned int value, cudaStream_t stream) {
    k_wait_counter<<<1, 1, 0, stream>>>(counter, value);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_pack_pixels(const float* rgb, void* out, int64_t npix, int format, cudaStream_t stream) {
    const int64_t work = format == RTGS_PIXELS_F16 ? (npix * 3 + 1) / 2 : npix;
    k_pack_pixels<<<(int)((work + 255) / 256), 256, 0, stream>>>(rgb, out, npix, format);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_add_counter(unsigned int* counter, cudaStream_t stream) {
    k_add_counter<<<1, 1, 0, stream>>>(counter);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_store_u32(unsigned int* counter, unsigned int value, cudaStream_t stream) {
    k_store_u32<<<1, 1, 0, stream>>>(counter, value);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}

int rtgs_launch_set_counter(unsigned int* counter, unsigned int value, cudaStream_t stream) {
    k_set_counter<<<1, 1, 0, stream>>>(counter, value);
    CUDA_TRY(cudaGetLastError());
    return RTGS_OK;
}
