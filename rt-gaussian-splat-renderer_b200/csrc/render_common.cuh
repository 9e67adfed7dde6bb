// render_common.cuh — declarations shared by the render kernels (sm_100a), all compiled in render.cu:
//   tile_lists.cuh lists_group    LBVH traversal, one candidate list per 4x8-pixel tile   (scene.py:406-450)
//   shade.cuh      shade_tile     intersection + k-buffer + SH compositing per tile       (gaussian.py:140-230,
//                                                                                          ray_tracer.py:79-104)
//   fused.cuh      k_render       the same path per tile with distance pruning (depth > 16, tiles whose list did
//                                 not fit the list pool, groups whose frustum holds ~1000 Gaussians or more)
//   render.cu      k_frame        ONE launch per frame: persistent warps alternate between lists_group and
//                                 shade_tile; k_tile_lists / k_shade_tiles are the same code as two launches
#pragma once
#include "common.cuh"
#include "gsmath.cuh"
#include <cuda_fp16.h>

namespace rtgs_dev {

constexpr int TILE_I = 4, TILE_J = 8;      // pixels per warp tile; lane = li * TILE_J + lj
constexpr int GROUP_TI = 2, GROUP_TJ = 2;  // tiles per traversal group: 8 x 16 pixels
constexpr int GPX_I = TILE_I * GROUP_TI, GPX_J = TILE_J * GROUP_TJ;
constexpr int MACRO_GI = 4, MACRO_GJ = 2;  // groups per 32x32-pixel macro tile (scheduling locality)
constexpr int TILES_PER_GROUP = GROUP_TI * GROUP_TJ;
constexpr int GROUPS_PER_MACRO = MACRO_GI * MACRO_GJ;
constexpr int TILES_PER_MACRO = TILES_PER_GROUP * GROUPS_PER_MACRO;
constexpr int MACRO_PX_I = GPX_I * MACRO_GI, MACRO_PX_J = GPX_J * MACRO_GJ;
constexpr int WARPS_PER_CTA = 8;
constexpr unsigned FULL = 0xffffffffu;

// Candidate lists (k_tile_lists -> k_shade_tiles): chunks of 32 ints in a global pool.  A chunk holds up
// to 31 sorted positions in [0..30] and the index of the NEXT chunk of the same tile in [31] (-1 = end).
// A tile's chunks are linked newest first: the head chunk holds the remainder ((count-1) % 31 + 1
// entries), every other chunk is full.
constexpr int CHUNK_IDS = 31;
constexpr int CHUNK_INTS = 32;
constexpr int SLAB_CHUNKS = 16;   // chunks a warp takes from the pool per atomic

struct TileDesc {
    int head;    // first chunk, -1 if the list is empty
    int count;   // candidates; -1: the list did not fit the pool, the tile is in the fallback list;
                 // | TILE_CAPPED: the list is depth-capped (heavy_lists.cuh), tile_cap[tile] holds the cap
};
constexpr int TILE_CAPPED = 1 << 30;

// CTR_FALLBACK / CTR_WORK3: tiles the traversal hands to k_render (list pool exhausted, or a group whose frustum holds
// too many candidates) and the cursor of the launch that renders them; CTR_FALLBACK2 / CTR_WORK4: tiles the shading
// hands over (three hits within rounding at the K-th place) and their cursor.  Two lists, because the first one is
// complete BEFORE the shading starts and its tiles are rendered concurrently with it (render.cu).
enum { CTR_WORK = 0, CTR_POOL = 1, CTR_FALLBACK = 2, CTR_WORK2 = 3, CTR_WORK3 = 4, CTR_DONE = 5, CTR_DONE2 = 6,
       CTR_FALLBACK2 = 7, CTR_WORK4 = 8, CTR_DONE3 = 9,
       CTR_HEAVY = 10, CTR_WORK5 = 11,   // heavy groups queued by the traversal / the cursor of k_heavy_lists
       CTR_HEAVY_FAILED = 12,            // ... of them handed on to k_render (statistics)
       CTR_COUNT = 16 };
enum { ST_RAYS = 0, ST_RAYS_HIT, ST_LAYERS, ST_NODES, ST_CANDS, ST_PAIRS, ST_F64, ST_TILES, ST_STEPS, ST_INSERTS,
       ST_FALLBACK, ST_USEFUL, ST_COUNT = 12,
       // high-water marks (maxima, not sums; statistics builds only): deepest traversal stacks and the fullest group
       // list seen - the stack bounds of tile_lists.cuh / fused.cuh checked on the device (compute-sanitizer is not
       // available on the GPU pool, so the deep-tree tests assert these instead)
       ST_MAX_LISTS_STACK = 12, ST_MAX_FUSED_STACK = 13, ST_MAX_GROUP_LIST = 14,
       // depth-capped lists (heavy_lists.cuh): groups listed that way, of them handed on to the fused kernel, cap raises,
       // candidates tested against the sample rays; ST_MAX_DEFERRED: longest deferred list (a maximum)
       ST_HEAVY_GROUPS = 15, ST_HEAVY_FAILED = 16, ST_HEAVY_PASSES = 17, ST_HEAVY_TESTS = 18, ST_MAX_DEFERRED = 19,
       ST_HEAVY_RETRIES = 20, ST_HEAVY_FAIL_LIST = 21, ST_HEAVY_FAIL_DEFER = 22, ST_HEAVY_FAIL_PASSES = 23,
       ST_HEAVY_CYC_WALK = 24, ST_HEAVY_CYC_TEST = 25, ST_HEAVY_CYC_PUBLISH = 26,   // warp clock cycles per phase
       ST_TOTAL = 32 };

struct RenderParams {
    const float4* nodes;
    const float4* nodes4;     // two-level nodes (k_tile_lists)
    const float4* geo;
    const float4* shp;
    cudaTextureObject_t geo_tex;   // (experiment SHADE_GEO_TEX) the geometry records as a linear float4 texture
    cudaTextureObject_t shp_tex;   // the same records as a linear float4 texture, or 0 (too many for one texture): eval_colour
                                   // fetches part of a record through the texture path, the rest with 256-bit loads
    const float4* raw;
    const float4* leafbox;
    CamD cam;
    int x0, y0, w, h;
    int macro_cols;  // macro tiles along j
    int stripe_mod, stripe_rem;   // render only macro-tile columns mi with mi % stripe_mod == stripe_rem (multi-GPU)
    int ntiles;      // macro_rows * macro_cols * TILES_PER_MACRO (tile ids, some outside the region)
    int depth;
    float t_cut;
    int accumulate, full_pitch, has_sh;
    float* out_rgb;
    float* out_T;
    unsigned int* counters;   // CTR_*: work counters of the three kernels, pool chunks taken, fallback tiles
    unsigned long long* stats;
    // candidate lists
    TileDesc* desc;           // ntiles
    int* pool;                // pool_chunks * CHUNK_INTS
    int pool_chunks;
    int* fallback_tiles;      // ntiles: tiles handed over by the traversal (lists_group)
    int* fallback_tiles2;     // ntiles: tiles handed over by the shading (shade_tile)
    int use_fallback_list;    // k_render: 0 = every tile of the region; bit 0 = the tiles of fallback_tiles, bit 1 =
                              // those of fallback_tiles2 (both: the first list, then the second)
    int early_trigger;        // k_render: let the next kernel on the stream start at once (programmatic dependent
                              // launch): the shading that follows does not depend on this launch
    int heavy_fused;          // k_tile_lists: a group whose list overflows shared memory goes to k_render (distance pruning)
    int heavy_limit;          // ... "overflows" = more candidates than this (<= the capacity of the shared-memory list)
    // depth-capped lists of heavy groups (heavy_lists.cuh; all unused while heavy_slab == 0)
    int heavy_slab;           // lists_group queues a group whose list overflows in heavy_groups instead (k_heavy_lists follows)
    int* heavy_groups;        // ngroups
    float* tile_cap;          // ntiles: every Gaussian that can enter a ray of the tile nearer than this is in its list
    int2* heavy_scratch;      // per warp of k_heavy_lists: 2 x heavy_defer_cap deferred (node, depth bits) entries
    int heavy_defer_cap;
    int slab_rank;            // the cap of a pass = the slab_rank-th smallest of the 32 per-lane nearest deferred depths
    int lists_single;         // lists_group pops one node per step while its stack holds more entries than this (tile_lists.cuh)
    // band completion (host-pipelined framebuffer copy, rtgs_render_host): the frame is cut into nbands bands of
    // band_macro_cols 32-pixel columns; a band is finished when all its tile ids have been rendered or skipped
    int nbands, band_macro_cols, macro_rows, schedule;
    unsigned int* band_done;  // device counters, one per band
    int* band_flags;          // mapped pinned host memory: set to 1 by the warp that finishes the band
    int* mirror;              // mapped pinned host memory: [0] list-pool demand of the frame, [1] a frame had fallback tiles
    // group publication (tile_lists.cuh -> shade.cuh inside one launch): ready[group] == seq <=> the descriptors and
    // list chunks of the group's four tiles are complete for THIS frame (no reset between frames)
    unsigned int* ready;
    unsigned int seq;
    // frame completion and multi-GPU hand-over (render.cu: finish_frame).  All optional (nullptr = off):
    //   arrive      counter the LAST CTA of the frame's last kernel release-increments at system scope once every store
    //               of the frame is performed; may live in a peer GPU's memory (tile / view sharding: the
    //               gathering rank waits for world x frames arrivals - no collective, no extra launch)
    //   grant       before a warp's first framebuffer store it waits until *grant >= grant_value (signed distance):
    //               the consumer of a peer-mapped framebuffer has released the buffer this frame is written into
    unsigned int* arrive;
    const unsigned int* grant;
    unsigned int grant_value;
    int tail_launch;          // k_frame: the last CTA launches the fused kernel for the fallback tiles itself
                              // (device-side tail launch) instead of the host queueing a third kernel per frame
    int final_kernel;         // this launch is the frame's last kernel: its last CTA completes the frame (frame_complete)
    int self_clean;           // ... and zeroes the work counters for the next frame (no memset between frames)
    int tail_grid;            // CTAs of a device-side k_render launch (2 per SM)
};

// System-scope hand-over of a framebuffer that other GPUs read or write (see RenderParams::grant).
struct PeerGrant {
    unsigned seen;
    bool ok;
};
__device__ __forceinline__ void grant_begin(const RenderParams& P, PeerGrant& g) {
    g.ok = P.grant == nullptr;
    g.seen = 0;
    // issued at kernel start, consumed before the warp's first store: normally satisfied long before
    if (!g.ok) asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(g.seen) : "l"(P.grant) : "memory");
}
__device__ __forceinline__ void grant_wait(const RenderParams& P, PeerGrant& g) {
    if (g.ok) return;
    while ((int)(g.seen - P.grant_value) < 0) {
        __nanosleep(500);
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(g.seen) : "l"(P.grant) : "memory");
    }
    g.ok = true;
}

// The frame is complete (call from ONE thread, after every CTA of the frame's last kernel has finished its stores):
// hand-over signal for whoever gathers the frame, then the work counters are zeroed for the next frame.
__device__ __forceinline__ void frame_complete(const RenderParams& P) {
    if (P.arrive)   // (the release covers everything cta_is_last has ordered before this thread)
        asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(P.arrive) : "memory");
    if (P.self_clean) {
#pragma unroll
        for (int k = 0; k < CTR_COUNT; ++k) P.counters[k] = 0u;
    }
}

// End of a kernel: count the finished CTAs; returns true in thread 0 of the CTA that finishes last, with every
// other CTA's stores ordered before it: each CTA's fence + atomic (device scope) synchronises with the last CTA's
// atomic + fence, and causality order is transitive across scopes, so only the ONE system-scope release in
// frame_complete is needed to publish all of them to another GPU (a system fence per CTA cost ~10 us per frame).
__device__ __forceinline__ bool cta_is_last(const RenderParams& P, int ctr) {
    __syncthreads();
    if (threadIdx.x != 0) return false;
    __threadfence();
    const unsigned prev = atomicAdd(P.counters + ctr, 1u);
    if (prev + 1u != gridDim.x) return false;
    __threadfence();
    return true;
}
__device__ __forceinline__ void cta_finish(const RenderParams& P, int ctr) {
    if (cta_is_last(P, ctr)) frame_complete(P);
}

// Descriptor of a published tile, read at L2: within one launch the line may have been cached in L1 while a
// neighbouring descriptor was still unwritten.
__device__ __forceinline__ TileDesc load_desc(const RenderParams& P, int tile) {
    const int2 v = __ldcg(reinterpret_cast<const int2*>(P.desc) + tile);
    TileDesc d;
    d.head = v.x;
    d.count = v.y;
    return d;
}


// Band completion (host-pipelined framebuffer copy, rtgs_render_host).  A tile id has been rendered (its framebuffer
// stores are issued) or skipped: it counts for its band, and the warp that completes a band raises the host-visible
// flag.  A warp's tiles come in order, so consecutive tiles nearly always belong to the same band: the counts are
// accumulated per warp (BandCount) and released in ONE atomic when the warp claims a tile of another band or ends -
// the release-add per tile (MEMBAR + ATOMG) cost k_shade_tiles 8 %.  The flush happens at CLAIM time, before the
// new tile is processed, so a band is never held back by the duration of a tile of the next band.
// The per-warp state {band, pending} lives in two ints of the warp's SHARED memory (only lane 0 touches them, and only
// in banded launches): in registers it cost the un-banded kernels 0.8 %.
struct BandCount {
    int* st;   // st[0] = band of the pending counts (-1: none), st[1] = pending count
};
__device__ __forceinline__ void band_begin(const RenderParams& P, BandCount& bc, int* smem2, int lane) {
    bc.st = smem2;
    if (P.nbands != 0 && lane == 0) {
        smem2[0] = -1;
        smem2[1] = 0;
    }
}
__device__ __forceinline__ int band_of(const RenderParams& P, int tile) {
    return (tile / TILES_PER_MACRO / P.macro_cols) / P.band_macro_cols;
}
// (lane 0 only)
__device__ __forceinline__ void band_flush_lane0(const RenderParams& P, BandCount& bc) {
    const unsigned pending = (unsigned)bc.st[1];
    if (pending != 0) {
        const int band = bc.st[0];
        const int cols = min(P.macro_rows, (band + 1) * P.band_macro_cols) - band * P.band_macro_cols;
        const unsigned total = (unsigned)(cols * P.macro_cols * TILES_PER_MACRO);
        // Release-add: the warp's framebuffer stores of all the counted tiles (ordered before it by the __syncwarp
        // that ends store_tile; release is cumulative) are visible before the count.  Only the warp that completes
        // the band pays for the acquire side.
        unsigned int before;
        asm volatile("atom.add.release.gpu.global.u32 %0, [%1], %2;"
                     : "=r"(before) : "l"(P.band_done + band), "r"(pending) : "memory");
        if (before + pending == total) {
            __threadfence();
            __threadfence_system();
            *reinterpret_cast<volatile int*>(P.band_flags + band) = 1;
        }
        bc.st[1] = 0;
    }
}
__device__ __forceinline__ void band_flush(const RenderParams& P, BandCount& bc, int lane) {
    if (P.nbands != 0 && lane == 0) band_flush_lane0(P, bc);
}
// call when a tile id has been claimed (before it is processed)
__device__ __forceinline__ void band_claim(const RenderParams& P, BandCount& bc, int tile, int lane) {
    if (P.nbands == 0 || lane != 0) return;
    const int band = band_of(P, tile);
    if (band != bc.st[0]) {
        band_flush_lane0(P, bc);
        bc.st[0] = band;
    }
}
// call with the whole warp converged, after store_tile (or when the tile is skipped)
__device__ __forceinline__ void tile_done(const RenderParams& P, BandCount& bc, int tile, int lane) {
    if (P.nbands != 0 && lane == 0) bc.st[1] += 1;
}

// 256-bit read-only global load (sm_100 LDG.E.256): the L1 data pipe is charged per 128-byte line and
// instruction, so a gather of 32-byte pieces costs half of what two 16-byte gathers do.  p is 32-byte aligned.
__device__ __forceinline__ void ldg256(const void* p, float4& a, float4& b) {
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
        : "l"(p));
}

// tile id -> pixel origin.  id = (macro * GROUPS_PER_MACRO + group) * TILES_PER_GROUP + sub, so that the
// four tiles of a traversal group are consecutive and consecutive groups share a 32x32-pixel macro tile.
// Order in which the macro-tile columns are scheduled (position -> column).  0: left to right (device renders:
// best locality and a cheap tail).  The banded framebuffer copy of rtgs_render_host wants bands to finish no
// faster than the DMA drains them at the END of the frame, so that nothing piles up behind the render:
// 1: from the image edges inwards (0, last, 1, last-1 ...; for a centred scene cheap columns first, expensive
// last); 2: rotated, the rightmost fifth first, then left to right.
__host__ __device__ __forceinline__ int macro_column(int macro_rows, int pos, int schedule) {
    if (schedule == 1) return (pos & 1) ? macro_rows - 1 - (pos >> 1) : (pos >> 1);
    if (schedule == 2) {
        const int head = macro_rows / 5;
        return pos < head ? macro_rows - head + pos : pos - head;
    }
    return pos;
}
__device__ __forceinline__ int macro_column(const RenderParams& P, int pos) {
    return macro_column(P.macro_rows, pos, P.schedule);
}

// Work item k of a launch -> tile / group id (>= `total` when the launch is exhausted).  per_col = ids per
// macro-tile column.  A stripe-sharded launch (RTGS_OPT_STRIPE) enumerates only the columns it owns: pulling
// and skipping the foreign ids costs an atomic round trip each, and with 7/8 of them foreign that was most of
// k_tile_lists at 8 GPUs.  (Banded launches and the rotated schedules keep the plain order: their band counters
// expect every id to be reported.)
__device__ __forceinline__ int work_to_id(const RenderParams& P, int k, int per_col, int total) {
    if (P.stripe_mod <= 1 || P.schedule != 0 || P.nbands > 0) return k;
    const int c = k / per_col;
    const int mi = P.stripe_rem + c * P.stripe_mod;
    return mi < P.macro_rows ? mi * per_col + (k - c * per_col) : total;
}

// Returns false for a group outside this launch's stripe (its macro-tile column belongs to another GPU).
__device__ __forceinline__ bool group_origin(const RenderParams& P, int group, int& gi0, int& gj0) {
    const int macro = group / GROUPS_PER_MACRO, lg = group % GROUPS_PER_MACRO;
    const int mi = macro_column(P, macro / P.macro_cols), mj = macro % P.macro_cols;
    gi0 = P.x0 + (mi * MACRO_GI + lg / MACRO_GJ) * GPX_I;
    gj0 = P.y0 + (mj * MACRO_GJ + lg % MACRO_GJ) * GPX_J;
    return P.stripe_mod <= 1 || mi % P.stripe_mod == P.stripe_rem;
}
__device__ __forceinline__ bool tile_origin(const RenderParams& P, int tile, int& i0, int& j0) {
    int gi0, gj0;
    const bool mine = group_origin(P, tile / TILES_PER_GROUP, gi0, gj0);
    const int sub = tile % TILES_PER_GROUP;
    i0 = gi0 + (sub / GROUP_TJ) * TILE_I;
    j0 = gj0 + (sub % GROUP_TJ) * TILE_J;
    return mine;
}

// ---- frustum of a pixel rectangle: 4 planes through the camera origin o, inward normals n[k]; a box
// (centre c, half size h) is outside plane k iff n.c + |n|.h - n.o < 0 ---------------------------------
struct Frustum {
    float nx[4], ny[4], nz[4];
    float ax[4], ay[4], az[4];   // |n|
    float d[4];                  // n.o
};

__device__ __forceinline__ void make_frustum(const CamD& cam, int il, int ih, int jl, int jh, Frustum& fr) {
    const double pxl = ((double)il - 0.5 * cam.W) * cam.ifx, pxh = ((double)ih - 0.5 * cam.W) * cam.ifx;
    const double pyl = ((double)jl - 0.5 * cam.H) * cam.ify, pyh = ((double)jh - 0.5 * cam.H) * cam.ify;
    d3 n[4];
    n[0] = cam_rot(cam, 1.0, 0.0, pxl);     // px >= pxl
    n[1] = cam_rot(cam, -1.0, 0.0, -pxh);   // px <= pxh
    n[2] = cam_rot(cam, 0.0, 1.0, pyl);     // py >= pyl
    n[3] = cam_rot(cam, 0.0, -1.0, -pyh);   // py <= pyh
    const float ox = (float)cam.o[0], oy = (float)cam.o[1], oz = (float)cam.o[2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        fr.nx[k] = (float)n[k].x; fr.ny[k] = (float)n[k].y; fr.nz[k] = (float)n[k].z;
        fr.ax[k] = fabsf(fr.nx[k]); fr.ay[k] = fabsf(fr.ny[k]); fr.az[k] = fabsf(fr.nz[k]);
        fr.d[k] = fr.nx[k] * ox + fr.ny[k] * oy + fr.nz[k] * oz;
    }
}

__device__ __forceinline__ bool box_in_frustum(const Frustum& f, float cx, float cy, float cz, float hx,
                                               float hy, float hz) {
    bool in = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float v = f.nx[k] * cx + f.ny[k] * cy + f.nz[k] * cz + f.ax[k] * hx + f.ay[k] * hy + f.az[k] * hz;
        in = in && (v >= f.d[k]);  // NaN / -inf (empty box) -> false
    }
    return in;
}

// Does the sqrt(3)-sigma ellipsoid of a Gaussian reach into the frustum?  Exact support function per plane:
// with u = n (.) h (h_i = sqrt(3 Sigma_ii)) and the correlation matrix C, the ellipsoid extends
// s = sqrt(u^T C u) along n, so it is outside plane k iff  n.p - n.o < -s.  (The box test uses the looser
// |u|_1 >= s.)  leaf = the 32-byte record k_pack writes: {p.xyz, h.x}{h.y, h.z, fp16 2rho_xy 2rho_xz, fp16 2rho_yz};
// the fp16 rounding of the correlations (<= 4.9e-4 absolute, i.e. <= 4.9e-4 |u|_1^2 <= 1.5e-3 |u|^2 in s^2) is
// covered by the factor 1.003 on the diagonal part.
__device__ __forceinline__ bool ellipsoid_in_frustum(const Frustum& f, const float4& la, const float4& lb) {
    const float2 r01 = __half22float2(*reinterpret_cast<const __half2*>(&lb.z));
    const float2 r2 = __half22float2(*reinterpret_cast<const __half2*>(&lb.w));
    bool in = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float dist = f.nx[k] * la.x + f.ny[k] * la.y + f.nz[k] * la.z - f.d[k];
        const float ux = f.nx[k] * la.w, uy = f.ny[k] * lb.x, uz = f.nz[k] * lb.y;
        const float s2 = 1.003f * (ux * ux + uy * uy + uz * uz) + ux * (uy * r01.x + uz * r01.y) + uy * uz * r2.x;
        in = in && (dist >= 0.0f || dist * dist <= s2);
    }
    return in;
}

// One plane of that test, two-sided: plane {x: n.x = d} through the camera origin; lo / hi = the ellipsoid
// reaches the side n.x >= d / the side n.x <= d.  A tile bounded by planes k (lower) and k+1 (upper) along an
// image axis is touched iff lo[k] && hi[k+1]; neighbouring tiles share the plane between them.
__device__ __forceinline__ void plane_side(float nx, float ny, float nz, float d, const float4& la, const float4& lb,
                                           const float2& r01, const float2& r2, bool& lo, bool& hi) {
    const float dist = nx * la.x + ny * la.y + nz * la.z - d;
    const float ux = nx * la.w, uy = ny * lb.x, uz = nz * lb.y;
    const float s2 = 1.003f * (ux * ux + uy * uy + uz * uz) + ux * (uy * r01.x + uz * r01.y) + uy * uz * r2.x;
    const bool reach = dist * dist <= s2;
    lo = dist >= 0.0f || reach;
    hi = dist <= 0.0f || reach;
}

// ---- per-ray box test of the stack traversals (k_trace_closest, k_render_backward) -----------------
// Entry distance of the ray (origin of, inverse direction idf) into the box [mn, mx], or +inf on a miss
// (bounding_box.py:50-89; hit iff t_min < t_max).  Float32 slabs inflated by a few ulp, so that rounding can never
// cull a true hit.
__device__ __forceinline__ float slab_entry(const float (&of)[3], const float (&idf)[3], const float (&mn)[3],
                                            const float (&mx)[3]) {
    float t0 = -INFINITY, t1 = INFINITY;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float ta = (mn[a] - of[a]) * idf[a], tb = (mx[a] - of[a]) * idf[a];
        float lo = fminf(ta, tb), hi = fmaxf(ta, tb);
        lo -= 4e-6f * fabsf(lo) + 1e-30f;
        hi += 4e-6f * fabsf(hi) + 1e-30f;
        if (ta != ta || tb != tb) { lo = -INFINITY; hi = INFINITY; }   // 0 * inf: ray inside slab plane
        t0 = fmaxf(t0, lo);
        t1 = fminf(t1, hi);
    }
    return (t0 <= t1) ? t0 : INFINITY;
}

// ---- float64 exact evaluation from raw parameters (rare path) ---------------------------------
__device__ __noinline__ static ExactHit exact_eval(const float4* __restrict__ raw, const CamD& cam, int s, int pi,
                                                   int pj) {
    float4 a = __ldg(raw + (int64_t)s * 3 + 0), b = __ldg(raw + (int64_t)s * 3 + 1),
           c = __ldg(raw + (int64_t)s * 3 + 2);
    double p[3] = {a.x, a.y, a.z};
    double q[4] = {a.w, b.x, b.y, b.z};
    double sc[3] = {b.w, c.x, c.y};
    d3 d = cam_dir(cam, (double)pi + 0.5, (double)pj + 0.5);
    return exact_intersect(p, q, sc, cam.o, d);
}

// Exact ordering of two hits of one ray whose float32 entry distances are within rounding of each
// other: float64 t1 from the raw parameters, ties broken by sorted position (rare path).
__device__ __noinline__ static bool exact_less(const float4* __restrict__ raw, const CamD& cam, int sa, int sb,
                                               int pi, int pj) {
    const ExactHit a = exact_eval(raw, cam, sa, pi, pj);
    const ExactHit b = exact_eval(raw, cam, sb, pi, pj);
    return a.t1 < b.t1 || (a.t1 == b.t1 && sa < sb);
}

// ---- SH basis, gaussian.py:149-163 (incl. the `5z^2 - 3z` term at :160 exactly as coded) ------
__device__ __forceinline__ void sh_basis(float x, float y, float z, float (&Y)[15]) {
    const float c0 = 0.9772050238058398f;   // sqrt(3/pi)
    const float c1 = 2.1850968611841584f;   // sqrt(15/pi)
    const float c2 = 1.2615662610100802f;   // sqrt(5/pi)
    const float c3 = 2.360174359706574f;    // sqrt(35/(2pi))
    const float c4 = 5.781222885281108f;    // sqrt(105/pi)
    const float c5 = 1.828183197857863f;    // sqrt(21/(2pi))
    const float c6 = 1.4927053303604616f;   // sqrt(7/pi)
    const float xx = x * x, yy = y * y, zz = z * z;
    Y[0] = 0.5f * c0 * y;
    Y[1] = 0.5f * c0 * z;
    Y[2] = 0.5f * c0 * x;
    Y[3] = 0.5f * c1 * x * y;
    Y[4] = 0.5f * c1 * y * z;
    Y[5] = 0.25f * c2 * (3.0f * zz - 1.0f);
    Y[6] = 0.5f * c1 * x * z;
    Y[7] = 0.25f * c1 * (xx - yy);
    Y[8] = 0.25f * c3 * y * (3.0f * xx - yy);
    Y[9] = 0.5f * c4 * x * y * z;
    Y[10] = 0.25f * c5 * y * (5.0f * zz - 1.0f);
    Y[11] = 0.25f * c6 * (5.0f * zz - 3.0f * z);
    Y[12] = 0.25f * c5 * x * (5.0f * zz - 1.0f);
    Y[13] = 0.25f * c4 * (xx - yy) * z;
    Y[14] = 0.25f * c3 * x * (xx - 3.0f * yy);
}

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Rays of one tile (float64 setup, camera.py:46-52).  Image-plane coordinates: px = (i + 0.5 - W/2)/fx.
// Tile centre (px0, py0); own offset (a, b) = (px - px0, py - py0).  UNNORMALISED directions are linear
// in (a, b):  D(a,b) = R (px0 + a, py0 + b, -1) = D0 + a Rx + b Ry;  the reference's direction is
// d = D / sqrt(px^2 + py^2 + 1); d0 likewise for the tile centre, d = d0 + delta.
struct TileRays {
    d3 D0, d0;
    double inv_d0d0;
    float dlx, dly, dlz;   // delta = d - d0
    float dnx, dny, dnz;   // normalize(d) for the SH basis (gaussian.py:200)
    float pa, pb;          // (a, b)
    float a_max, b_max, dl_max;
};

__device__ __forceinline__ void make_tile_rays(const CamD& cam, int i0, int j0, int pi, int pj, bool active,
                                               TileRays& r) {
    const double px0 = ((double)i0 + 0.5 * TILE_I - 0.5 * cam.W) * cam.ifx;
    const double py0 = ((double)j0 + 0.5 * TILE_J - 0.5 * cam.H) * cam.ify;
    r.D0 = cam_rot(cam, px0, py0, -1.0);
    const double n0 = rsqrt(px0 * px0 + py0 * py0 + 1.0);
    r.d0 = d3make(r.D0.x * n0, r.D0.y * n0, r.D0.z * n0);
    r.inv_d0d0 = 1.0 / d3dot(r.d0, r.d0);
    const double ad = active ? ((double)(pi - i0) + 0.5 - 0.5 * TILE_I) * cam.ifx : 0.0;
    const double bd = active ? ((double)(pj - j0) + 0.5 - 0.5 * TILE_J) * cam.ify : 0.0;
    {
        const double px = px0 + ad, py = py0 + bd;
        const double nn = rsqrt(px * px + py * py + 1.0);
        const d3 dw = d3make((r.D0.x + ad * cam.R[0] + bd * cam.R[1]) * nn, (r.D0.y + ad * cam.R[3] + bd * cam.R[4]) * nn,
                             (r.D0.z + ad * cam.R[6] + bd * cam.R[7]) * nn);
        r.dlx = (float)(dw.x - r.d0.x); r.dly = (float)(dw.y - r.d0.y); r.dlz = (float)(dw.z - r.d0.z);
        const double il = rsqrt(d3dot(dw, dw));
        r.dnx = (float)(dw.x * il); r.dny = (float)(dw.y * il); r.dnz = (float)(dw.z * il);
    }
    r.pa = (float)ad;
    r.pb = (float)bd;
    r.a_max = (float)(0.5 * TILE_I * fabs(cam.ifx));
    r.b_max = (float)(0.5 * TILE_J * fabs(cam.ify));
    float m = sqrtf(r.dlx * r.dlx + r.dly * r.dly + r.dlz * r.dlz);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, o));
    r.dl_max = m;
}

// Per-(tile, candidate) staging in float64 by one lane: the precise record (origin shifted to the
// closest point of the tile-centre ray) and the coarse quadratic.
//   rec: {W00 W01 W02 W10} {W11 W12 W20 W21} {W22 e0.xyz} {g0.xyz t_c} {opacity, s, band, t_lo}
//   poly: S(a,b) = c0 + a (c1 + a c3 + b c4) + b (c2 + b c5) < 0  <=>  possibly q < 3 + band
// With o' = W (o - p) = -W v and G(a,b) = W D(a,b) = G0 + a Gx + b Gy:
//   q(a,b) = |o' x G|^2 / |G|^2 = N/Dn,  m = o' x G = M0 + a Mx + b My,
//   S = N - (3 + band) Dn - margin, margin bounding the float32 evaluation error.
template <bool WITH_T_LO = false>
__device__ __forceinline__ void stage_candidate(const RenderParams& P, const TileRays& tr, int s, float4 (&rec)[5],
                                                float (&poly)[6]) {
    const CamD& cam = P.cam;
    float4 g0, g1, g2, g3;
#if SHADE_GEO_TEX
    {   // experiment: the 64-byte geometry record through the texture path as well
        const int t0 = s * 4;
        g0 = tex1Dfetch<float4>(P.geo_tex, t0); g1 = tex1Dfetch<float4>(P.geo_tex, t0 + 1);
        g2 = tex1Dfetch<float4>(P.geo_tex, t0 + 2); g3 = tex1Dfetch<float4>(P.geo_tex, t0 + 3);
    }
#else
    ldg256(P.geo + (int64_t)s * 4 + 0, g0, g1);
    ldg256(P.geo + (int64_t)s * 4 + 2, g2, g3);
#endif
    const double W00 = g1.x, W01 = g1.y, W02 = g1.z, W10 = g1.w, W11 = g2.x, W12 = g2.y, W20 = g2.z, W21 = g2.w,
                 W22 = g3.x;
    auto Wmul = [&](const d3& v) {
        return d3make(W00 * v.x + W01 * v.y + W02 * v.z, W10 * v.x + W11 * v.y + W12 * v.z,
                      W20 * v.x + W21 * v.y + W22 * v.z);
    };
    const d3 v = d3make((double)g0.x - cam.o[0], (double)g0.y - cam.o[1], (double)g0.z - cam.o[2]);
    const double tc = d3dot(v, tr.d0) * tr.inv_d0d0;
    const d3 e0 = Wmul(d3make(tc * tr.d0.x - v.x, tc * tr.d0.y - v.y, tc * tr.d0.z - v.z));
    const d3 gd = Wmul(tr.d0);
    const float wn = sqrtf(g1.x * g1.x + g1.y * g1.y + g1.z * g1.z + g1.w * g1.w + g2.x * g2.x + g2.y * g2.y +
                           g2.z * g2.z + g2.w * g2.w + g3.x * g3.x);
    const float eb = (float)sqrt(d3dot(e0, e0)) + fabsf((float)tc) * tr.dl_max * wn;
    const float band = 4e-6f * (3.0f + eb * eb);
    rec[0] = g1;
    rec[1] = g2;
    rec[2] = make_float4(g3.x, (float)e0.x, (float)e0.y, (float)e0.z);
    rec[3] = make_float4((float)gd.x, (float)gd.y, (float)gd.z, (float)tc);
    // lower bound of the entry distance for every ray of the tile: t1 = tc + tau with
    // |tau| <= (|e| + sqrt 3) / |W d|, |e| <= eb (above) and |W d| >= |W d0| - |W| |delta|max
    // (only the fused kernel uses it: it prunes per ray by distance)
    float t_lo = -INFINITY;
    if (WITH_T_LO) {
        const float gn = (float)sqrt(d3dot(gd, gd)) - wn * tr.dl_max;
        if (gn > 0.0f) t_lo = __double2float_rd(tc - (double)((eb + 1.7320509f) / gn) * 1.000001);
    }
    rec[4] = make_float4(g0.w, __int_as_float(s), band, t_lo);
    const d3 op = Wmul(d3make(-v.x, -v.y, -v.z));
    const d3 G0 = Wmul(tr.D0);
    const d3 Gx = Wmul(d3make(cam.R[0], cam.R[3], cam.R[6]));
    const d3 Gy = Wmul(d3make(cam.R[1], cam.R[4], cam.R[7]));
    const d3 M0 = d3cross(op, G0), Mx = d3cross(op, Gx), My = d3cross(op, Gy);
    const double lim = 3.0 + (double)band;
    const double m00 = d3dot(M0, M0), m0x = d3dot(M0, Mx), m0y = d3dot(M0, My), mxx = d3dot(Mx, Mx),
                 mxy = d3dot(Mx, My), myy = d3dot(My, My);
    const double g00 = lim * d3dot(G0, G0), g0x = lim * d3dot(G0, Gx), g0y = lim * d3dot(G0, Gy),
                 gxx = lim * d3dot(Gx, Gx), gxy = lim * d3dot(Gx, Gy), gyy = lim * d3dot(Gy, Gy);
    const double am = tr.a_max, bm = tr.b_max;
    // magnitude of the terms BEFORE cancellation (N and Dn parts separately)
    const double E = m00 + g00 + 2.0 * am * (fabs(m0x) + fabs(g0x)) + 2.0 * bm * (fabs(m0y) + fabs(g0y)) +
                     am * am * (mxx + gxx) + 2.0 * am * bm * (fabs(mxy) + fabs(gxy)) + bm * bm * (myy + gyy);
    poly[0] = (float)(m00 - g00 - 2e-6 * E);
    poly[1] = (float)(2.0 * (m0x - g0x));
    poly[2] = (float)(2.0 * (m0y - g0y));
    poly[3] = (float)(mxx - gxx);
    poly[4] = (float)(2.0 * (mxy - gxy));
    poly[5] = (float)(myy - gyy);
}

__device__ __forceinline__ bool coarse_test(const float (&p)[6], float pa, float pb) {
    const float ta = fmaf(pa, p[3], fmaf(pb, p[4], p[1]));   // c1 + a c3 + b c4
    const float tb = fmaf(pb, p[5], p[2]);                   // c2 + b c5
    return fmaf(pa, ta, fmaf(pb, tb, p[0])) < 0.0f;
}

// The precise per-ray test of one staged candidate (float32 relative to the tile-centre ray, decisions
// within the band re-evaluated in float64): hit?, entry distance t1, alpha = opacity * exp(-q).
struct PreciseHit {
    bool hit;
    float t1, alpha;
    int s;
    bool refined;
};

__device__ __forceinline__ PreciseHit precise_test(const RenderParams& P, const float4* rc, float dlx, float dly,
                                                   float dlz, int pi, int pj) {
    const float4 r0 = rc[0], r1 = rc[1], r2 = rc[2], r3 = rc[3], ax = rc[4];
    const float wx = r0.x * dlx + r0.y * dly + r0.z * dlz;
    const float wy = r0.w * dlx + r1.x * dly + r1.y * dlz;
    const float wz = r1.z * dlx + r1.w * dly + r2.x * dlz;
    const float tc = r3.w;
    const float dx = r3.x + wx, dy = r3.y + wy, dz = r3.z + wz;                 // d' = W d
    const float ex = r2.y + tc * wx, ey = r2.z + tc * wy, ez = r2.w + tc * wz;  // W (r(tc) - p)
    const float A = dx * dx + dy * dy + dz * dz;
    const float Bh = ex * dx + ey * dy + ez * dz;
    const float mx = ey * dz - ez * dy, my = ez * dx - ex * dz, mz = ex * dy - ey * dx;
    const float iA = rcp_approx(A);
    float q = (mx * mx + my * my + mz * mz) * iA;   // min Mahalanobis^2 along the ray
    // tau = -Bh/A - sqrt((3 - q)/A)  (near root relative to tc)
    const float tau = -Bh * iA - sqrt_approx(fmaxf(3.0f - q, 0.0f) * iA);
    PreciseHit h;
    h.t1 = tc + tau;
    h.s = __float_as_int(ax.y);
    h.hit = (q < 3.0f) && (h.t1 > 0.0f);
    h.refined = false;
    const bool near_q = fabsf(q - 3.0f) < ax.z;
    // t1 = tc + tau loses its float32 accuracy where the two terms cancel (a camera just outside a large ellipsoid:
    // tc = 0.5, tau = -0.4992 - two such hits 5e-8 apart were composited in the wrong order).  Where the entry
    // distance is smaller than |tau| it is taken from the float64 evaluation, so that every kept distance is accurate
    // relative to ITSELF and the relative tie bands of the k-buffer hold (elsewhere its error is <= 6e-7 t1).
    // Distances that are negative beyond rounding - the camera inside the ellipsoid - are misses either way.
    const bool near_t = (q < 3.0f + ax.z) && h.t1 > -2e-6f * (fabsf(tc) + fabsf(tau)) && h.t1 < fabsf(tau);
    if (near_q || near_t) {
        const ExactHit e = exact_eval(P.raw, P.cam, h.s, pi, pj);
        h.hit = e.hit && (e.t1 > 0.0);
        q = (float)e.q;
        h.t1 = (float)e.t1;
        h.refined = true;
    }
    h.alpha = ax.x * __expf(-q);   // opacity * exp(-q)  (gaussian.py:197-198)
    return h;
}

#ifndef SHADE_SH_TEX
#define SHADE_SH_TEX 8     // quads (of 12) of an SH record fetched through the texture path; even.  Measured on the
#endif                     // bench scene (k_shade_tiles): 0 -> 0.585 ms, 4 -> 0.554, 6 -> 0.544, 8 -> 0.536, 10 -> 0.537, 12 -> 0.551
#ifndef SHADE_GEO_TEX
#define SHADE_GEO_TEX 0
#endif
#ifndef SHADE_SH_TEX_RUNTIME
#define SHADE_SH_TEX_RUNTIME 1   // 1: scenes too large for one linear texture fall back to loads at run time (P.shp_tex == 0)
#endif
constexpr long long SH_TEX_MAX_RECORDS = (1ll << 27) / 12;   // one linear texture holds 2^27 texels
static_assert(SHADE_SH_TEX >= 0 && SHADE_SH_TEX <= 12 && SHADE_SH_TEX % 2 == 0, "SHADE_SH_TEX: even, 0..12");
// rgb = color + eval_sh(normalize(dir))  (gaussian.py:199-200) of the Gaussian at sorted position s.
// With SH the 192-byte record holds the 45 coefficients followed by the DC colour.
__device__ __forceinline__ void eval_colour(const RenderParams& P, int s, const float (&Y)[15], float& r, float& g,
                                            float& b) {
    if (P.has_sh) {
        const float4* sp = P.shp + (int64_t)s * 12;
        float v[48];
        // The record comes in through BOTH L1 front ends: the first SHADE_SH_TEX quads as 16-byte texture fetches (TEX
        // pipe, a linear float4 texture over the same memory; tex1Dfetch is cheaper than a 2-D fetch: 0.536 vs 0.560 ms),
        // the rest as 256-bit loads (LSU pipe).  The LSU pipe is what bounds the shading (shared-memory gathers + these
        // loads: 85 % busy before); the texture path has wavefront throughput of its own.  The handle must be
        // warp-uniform (a per-lane choice among several textures made the fetches 35 % slower than no texture at
        // all), so scenes beyond one linear texture (2^27 texels = 11 M records) take the all-LSU path.
#if SHADE_SH_TEX_RUNTIME
        if (P.shp_tex == 0) {
#pragma unroll
            for (int f = 0; f < SHADE_SH_TEX / 2; ++f) {
                float4 x, y;
                ldg256(sp + 2 * f, x, y);
                v[8 * f] = x.x; v[8 * f + 1] = x.y; v[8 * f + 2] = x.z; v[8 * f + 3] = x.w;
                v[8 * f + 4] = y.x; v[8 * f + 5] = y.y; v[8 * f + 6] = y.z; v[8 * f + 7] = y.w;
            }
        } else
#endif
        {
#pragma unroll
            for (int f = 0; f < SHADE_SH_TEX; ++f) {
                const float4 x = tex1Dfetch<float4>(P.shp_tex, s * 12 + f);
                v[4 * f] = x.x; v[4 * f + 1] = x.y; v[4 * f + 2] = x.z; v[4 * f + 3] = x.w;
            }
        }
#pragma unroll
        for (int f = SHADE_SH_TEX / 2; f < 6; ++f) {
            float4 x, y;
            ldg256(sp + 2 * f, x, y);
            v[8 * f] = x.x; v[8 * f + 1] = x.y; v[8 * f + 2] = x.z; v[8 * f + 3] = x.w;
            v[8 * f + 4] = y.x; v[8 * f + 5] = y.y; v[8 * f + 6] = y.z; v[8 * f + 7] = y.w;
        }
        r = v[45]; g = v[46]; b = v[47];
#pragma unroll
        for (int j = 0; j < 15; ++j) {
            r = fmaf(Y[j], v[3 * j + 0], r);
            g = fmaf(Y[j], v[3 * j + 1], g);
            b = fmaf(Y[j], v[3 * j + 2], b);
        }
    } else {
        const float4 g3 = __ldg(P.geo + (int64_t)s * 4 + 3);
        r = g3.y; g = g3.z; b = g3.w;
    }
}

// Framebuffer write of one tile: staged through `ob` (>= 96 floats of shared memory) so that every store
// instruction covers whole 32-byte sectors (each tile column is 8 pixels = 96 contiguous bytes).
__device__ __forceinline__ void store_tile(const RenderParams& P, float* ob, int lane, int i0, int j0, int pi, int pj,
                                           bool active, float cr, float cg, float cb, float T) {
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
    __syncwarp();
    ob[lane * 3 + 0] = cr;
    ob[lane * 3 + 1] = cg;
    ob[lane * 3 + 2] = cb;
    __syncwarp();
    const int pitch = P.full_pitch ? P.cam.H : P.h;
    const int bi = P.full_pitch ? 0 : P.x0, bj = P.full_pitch ? 0 : P.y0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int f = r * 32 + lane;
        const int row = f / (3 * TILE_J), col = f % (3 * TILE_J);
        const int qi = i0 + row, qj = j0 + col / 3;
        if (qi < xe && qj < ye) {
            float* o = P.out_rgb + ((int64_t)(qi - bi) * pitch + (j0 - bj)) * 3 + col;
            if (P.accumulate) *o += ob[f];
            else *o = ob[f];
        }
    }
    if (active && P.out_T) P.out_T[(int64_t)(pi - bi) * pitch + (pj - bj)] = T;
    __syncwarp();   // every lane's RGB and T stores are ordered before whatever lane 0 releases next (tile_done)
}

}  // namespace rtgs_dev

