// tile_lists.cuh — the BVH traversal of the render path (scene.py:406-450), done once per frame for whole
// pixel tiles instead of once per ray and per compositing step.  Device code shared by the stand-alone
// k_tile_lists kernel and the single-launch frame kernel k_frame (render.cu).
//
// All primary rays share the camera origin, so a rectangle of pixels is a thin pyramid bounded by 4 planes
// through the origin, and "every Gaussian whose bound some ray of the rectangle hits" is a frustum query on the
// LBVH.  A warp owns one 8x16-pixel GROUP at a time:
//   1. group traversal - nodes are popped from a shared-memory stack in batches; every popped node is a
//      two-level record (lbvh.cu: k_pack_nodes4: the 64-byte records of both children side by side), so one step
//      descends two tree levels; the grandchild boxes are tested against the 4 planes and the survivors compacted
//      with ballot/popc (internal -> stack, leaves -> the group's candidate list in shared memory).
//      LISTS_NODES_PER_STEP = 16: a PAIR of lanes shares a node (lane parity picks the child record);
//      LISTS_NODES_PER_STEP = 32: every lane takes a whole node (both records, four boxes): half as many
//      dependent steps per group, which is what bounds a frame that is spread over many GPUs (few groups per SM);
//   2. the list is filtered for the group's four 4x8-pixel tiles at once - the 2x2 tiles are bounded by 3 + 3
//      planes, one 32-byte leaf record per lane, six exact ellipsoid-vs-plane support tests decide all four tiles
//      - and streamed to the global list pool in 128-byte chunks (render_common.cuh), where shade_tile picks it up.
// A group whose list would overflow shared memory goes to the fused kernel (fused.cuh), which traverses near first
// and prunes by distance; a tile whose list does not fit the pool is handed to it too.  Nothing is ever dropped.
//
// When the four descriptors of a group are written the group is PUBLISHED: ready[group] = frame sequence number
// (release).  In the single-launch frame kernel the shading warps acquire that flag, so traversal and shading of
// one frame overlap inside one kernel; the stand-alone kernels do not need it (kernel boundary).
#pragma once
#include "render_common.cuh"

namespace rtgs_dev {

constexpr int LISTS_NODES_PER_STEP = 16;
constexpr int LISTS_TAKE = LISTS_NODES_PER_STEP;
static_assert(LISTS_TAKE == 16 || LISTS_TAKE == 32, "nodes per traversal step: 16 (lane pair per node) or 32");

// Stack bound.  A batch step pops `take` two-level nodes and pushes <= 4 grandchildren each: growth <= 3 * take.
// Above P.lists_single entries one node is popped per step (depth first): growth <= 3 per two-level step, i.e.
// <= 3 * ceil(depth / 2) over a whole descent, `depth` being the depth of the scene's deepest leaf (measured by
// the build, lbvh.cu: k_max_depth; <= RTGS_MAX_TREE_DEPTH).  The host sets
//   lists_single = min(LISTS_SINGLE, LISTS_STACK_CAP - 3 * LISTS_TAKE - 3 * ceil(depth / 2))    (render.cu)
// so the stack cannot overflow whatever the tree looks like; shallow trees (every real scene: ~30 levels for 1 M
// Gaussians) get the batch threshold that is fastest (LISTS_SINGLE), the deepest possible tree degrades to
// depth-first early.
constexpr int LISTS_SINGLE = 112;
constexpr int LISTS_STACK_ENTRIES = 256;
constexpr int LISTS_STACK_CAP = LISTS_STACK_ENTRIES;
static_assert(LISTS_STACK_CAP - 3 * LISTS_TAKE - 3 * ((RTGS_MAX_TREE_DEPTH + 1) / 2) >= 4,
              "lists_group: stack too small for the deepest tree");
__host__ __device__ constexpr int lists_single_bound(int tree_depth) {
    return LISTS_STACK_CAP - 3 * LISTS_TAKE - 3 * ((tree_depth + 1) / 2);
}
constexpr int GLIST_CAP = 960;
constexpr int CQ_TILE = 64;                          // per-tile output queue of the fused four-tile filter (< 31 + 32)
constexpr int CQ_CAP = TILES_PER_GROUP * CQ_TILE;    // the per-tile traversal uses it as one queue
static_assert(TILES_PER_GROUP == 4, "lists_group: the second-chunk test is written for four tiles");
static_assert(GLIST_CAP >= LISTS_STACK_CAP, "per-tile traversal keeps its stack in the group list");
static_assert(CQ_CAP >= CHUNK_IDS + 4 * LISTS_TAKE, "per-tile traversal: a step may add 4 leaves per node");

struct __align__(16) ListsShared {
    int stack[LISTS_STACK_CAP];
    int glist[GLIST_CAP];
    int cq[CQ_CAP];
};

// per-warp state that lives across groups: the slab of pool chunks the warp owns, and its counters
struct ListsState {
    int slab_next = 0, slab_end = 0;
    unsigned long long st_nodes = 0, st_steps = 0, st_cands = 0;
    unsigned st_max_stack = 0, st_max_list = 0;     // high-water marks (statistics builds)
    bool heavy_flagged = false;                     // this warp has reported a heavy group to the host (mirror[2])
};

// `group` is a group of this launch whose pixel origin (gi0, gj0) lies inside the rendered region (the caller has
// checked group_origin: nobody waits for any other group).
template <bool STATS>
__device__ __forceinline__ void lists_group(const RenderParams& P, ListsShared& ws, ListsState& S, int group, int gi0,
                                            int gj0, int lane) {
    const unsigned lt_mask = (1u << lane) - 1u;
    const CamD& cam = P.cam;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
#define ST(expr) do { if (STATS) { expr; } } while (0)

    // one traversal step, two tree levels deep (see the header comment)
    auto traverse_step = [&](int* stk, int& top, int* dst, int& nd, const Frustum& fr) {
        const int take = top > P.lists_single ? 1 : min(LISTS_TAKE, top);
        if constexpr (LISTS_TAKE == 16) {
            // a PAIR of lanes shares a node; lane parity picks the record of its left or right child
            int node = -1;
            if ((lane >> 1) < take) node = stk[top - 1 - (lane >> 1)];
            top -= take;
            __syncwarp();
            bool h0 = false, h1 = false;
            int c0 = 0, c1 = 0;
            if (node >= 0) {
                const float4* rec = P.nodes4 + (int64_t)node * 8 + (lane & 1) * 4;
                float4 a, b, c, d;
                ldg256(rec + 0, a, b);
                ldg256(rec + 2, c, d);
                c0 = __float_as_int(d.x);
                c1 = __float_as_int(d.y);
                h0 = box_in_frustum(fr, a.x, a.y, a.z, a.w, b.x, b.y);
                h1 = box_in_frustum(fr, b.z, b.w, c.x, c.y, c.z, c.w);
            }
            ST(S.st_nodes += 4ull * (unsigned)take);
            ST(S.st_steps += 1);
            const unsigned mI0 = __ballot_sync(FULL, h0 && c0 >= 0), mI1 = __ballot_sync(FULL, h1 && c1 >= 0);
            const unsigned mL0 = __ballot_sync(FULL, h0 && c0 < 0), mL1 = __ballot_sync(FULL, h1 && c1 < 0);
            if (h0 && c0 >= 0) stk[top + __popc(mI0 & lt_mask)] = c0;
            const int topa = top + __popc(mI0);
            if (h1 && c1 >= 0) stk[topa + __popc(mI1 & lt_mask)] = c1;
            top = topa + __popc(mI1);
            if (h0 && c0 < 0) dst[nd + __popc(mL0 & lt_mask)] = ~c0;
            const int nda = nd + __popc(mL0);
            if (h1 && c1 < 0) dst[nda + __popc(mL1 & lt_mask)] = ~c1;
            nd = nda + __popc(mL1);
            __syncwarp();
        } else {
            // every lane takes a whole two-level node: both child records, four grandchild boxes
            int node = -1;
            if (lane < take) node = stk[top - 1 - lane];
            top -= take;
            __syncwarp();
            bool hit[4];
            int ch[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) { hit[k] = false; ch[k] = 0; }
            if (node >= 0) {
                const float4* rec = P.nodes4 + (int64_t)node * 8;
                float4 q[8];
#pragma unroll
                for (int k = 0; k < 4; ++k) ldg256(rec + 2 * k, q[2 * k], q[2 * k + 1]);   // all four loads in flight
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float4 a = q[4 * h], b = q[4 * h + 1], c = q[4 * h + 2], d = q[4 * h + 3];
                    ch[2 * h] = __float_as_int(d.x);
                    ch[2 * h + 1] = __float_as_int(d.y);
                    hit[2 * h] = box_in_frustum(fr, a.x, a.y, a.z, a.w, b.x, b.y);
                    hit[2 * h + 1] = box_in_frustum(fr, b.z, b.w, c.x, c.y, c.z, c.w);
                }
            }
            ST(S.st_nodes += 4ull * (unsigned)take);
            ST(S.st_steps += 1);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool in = hit[k] && ch[k] >= 0;
                const unsigned m = __ballot_sync(FULL, in);
                if (in) stk[top + __popc(m & lt_mask)] = ch[k];
                top += __popc(m);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool lf = hit[k] && ch[k] < 0;
                const unsigned m = __ballot_sync(FULL, lf);
                if (lf) dst[nd + __popc(m & lt_mask)] = ~ch[k];
                nd += __popc(m);
            }
            __syncwarp();
        }
    };

    // take one chunk from the pool (-1: exhausted)
    auto alloc_chunk = [&]() -> int {
        if (S.slab_next == S.slab_end) {
            unsigned base = 0;
            if (lane == 0) base = atomicAdd(P.counters + CTR_POOL, (unsigned)SLAB_CHUNKS);
            base = __shfl_sync(FULL, base, 0);
            if (base + (unsigned)SLAB_CHUNKS > (unsigned)P.pool_chunks) return -1;
            S.slab_next = (int)base;
            S.slab_end = S.slab_next + SLAB_CHUNKS;
        }
        return S.slab_next++;
    };

    // write the last `m` entries of q as one chunk linked in front of `head`
    auto write_chunk = [&](const int* q, int m, int& ncq, int& head, int& count) -> bool {
        const int chunk = alloc_chunk();
        if (chunk < 0) return false;
        int v = head;
        if (lane < m) v = q[ncq - m + lane];
        if (lane < m || lane == CHUNK_INTS - 1) P.pool[(int64_t)chunk * CHUNK_INTS + lane] = v;
        head = chunk;
        ncq -= m;
        count += m;
        __syncwarp();
        return true;
    };

    // ---- group traversal: the LBVH once for the 8x16-pixel frustum ---------------------------
    int ng = 0;
    bool per_tile = false;
    {
        Frustum fg;
        make_frustum(cam, gi0, min(gi0 + GPX_I, xe), gj0, min(gj0 + GPX_J, ye), fg);
        int top = 1;
        if (lane == 0) ws.stack[0] = 0;
        __syncwarp();
#pragma unroll 1
        while (top > 0) {
            if (ng > min(GLIST_CAP - 4 * LISTS_TAKE, P.heavy_limit)) {   // too many candidates for the shared list
                per_tile = true;
                break;
            }
            traverse_step(ws.stack, top, ws.glist, ng, fg);
            ST(S.st_max_stack = max(S.st_max_stack, (unsigned)top));
            ST(S.st_max_list = max(S.st_max_list, (unsigned)ng));
        }
    }

    // a tile's list is complete: descriptor, or the fallback list if the pool ran out
    auto finish_tile = [&](int tile, int head, int count, bool ok) {
        if (lane == 0) {
            TileDesc d;
            d.head = head;
            d.count = ok ? count : -1;
            P.desc[tile] = d;
            if (!ok) P.fallback_tiles[atomicAdd(P.counters + CTR_FALLBACK, 1u)] = tile;
        }
        ST(S.st_cands += ok ? (unsigned)count : 0u);
    };

    if (!per_tile) {
        // ---- fused filter of the group's candidates for its four tiles ------------------------------
        // The 2x2 tiles are bounded by 3 + 3 planes through the camera origin (pixel edges gi0, +4, +8 and
        // gj0, +8, +16); a plane serves the tile on either side, so six exact support tests per Gaussian
        // (render_common.cuh: plane_side) decide all four tiles, and every leaf record is fetched once.
        float pnx[6], pny[6], pnz[6], pd[6];
        {
            const float ox = (float)cam.o[0], oy = (float)cam.o[1], oz = (float)cam.o[2];
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                d3 n;
                if (k < 3) n = cam_rot(cam, 1.0, 0.0, ((double)(gi0 + k * TILE_I) - 0.5 * cam.W) * cam.ifx);
                else n = cam_rot(cam, 0.0, 1.0, ((double)(gj0 + (k - 3) * TILE_J) - 0.5 * cam.H) * cam.ify);
                pnx[k] = (float)n.x; pny[k] = (float)n.y; pnz[k] = (float)n.z;
                pd[k] = pnx[k] * ox + pny[k] * oy + pnz[k] * oz;
            }
        }
        int head[TILES_PER_GROUP], count[TILES_PER_GROUP], ncq[TILES_PER_GROUP];
        bool ok[TILES_PER_GROUP], valid[TILES_PER_GROUP];
#pragma unroll
        for (int t = 0; t < TILES_PER_GROUP; ++t) {
            head[t] = -1; count[t] = 0; ncq[t] = 0; ok[t] = true;
            valid[t] = gi0 + (t / GROUP_TJ) * TILE_I < xe && gj0 + (t % GROUP_TJ) * TILE_J < ye;
        }
#pragma unroll 1
        for (int gpos = 0; gpos < ng; gpos += 32) {
            const int idx = gpos + lane;
            int s = 0;
            bool lo[6], hi[6];   // the ellipsoid reaches the >= side / the <= side of plane k
#pragma unroll
            for (int k = 0; k < 6; ++k) lo[k] = hi[k] = false;
            if (idx < ng) {
                s = ws.glist[idx];
                float4 a, b;
                ldg256(P.leafbox + (int64_t)s * 2, a, b);
                const float2 r01 = __half22float2(*reinterpret_cast<const __half2*>(&b.z));
                const float2 r2 = __half22float2(*reinterpret_cast<const __half2*>(&b.w));
#pragma unroll
                for (int k = 0; k < 6; ++k)
                    plane_side(pnx[k], pny[k], pnz[k], pd[k], a, b, r01, r2, lo[k], hi[k]);
            }
            ST(S.st_nodes += (unsigned)min(32, ng - gpos));
            ST(S.st_steps += 1);
#pragma unroll
            for (int t = 0; t < TILES_PER_GROUP; ++t) {
                const int ta = t / GROUP_TJ, tb = 3 + t % GROUP_TJ;
                const bool h = valid[t] && ok[t] && lo[ta] && hi[ta + 1] && lo[tb] && hi[tb + 1];
                const unsigned mh = __ballot_sync(FULL, h);
                if (h) ws.cq[t * CQ_TILE + ncq[t] + __popc(mh & lt_mask)] = s;
                ncq[t] += __popc(mh);
            }
            __syncwarp();
            // (a batch may add 32 entries to a queue that holds up to 30: two chunks then, or the queue would creep
            // past its 64 slots into its neighbour's - a dense cluster of Gaussians that all touch one tile)
#pragma unroll
            for (int t = 0; t < TILES_PER_GROUP; ++t)
                if (ncq[t] >= CHUNK_IDS) ok[t] = write_chunk(ws.cq + t * CQ_TILE, CHUNK_IDS, ncq[t], head[t], count[t]);
            if (max(max(ncq[0], ncq[1]), max(ncq[2], ncq[3])) >= CHUNK_IDS) {   // rare: a second chunk
#pragma unroll
                for (int t = 0; t < TILES_PER_GROUP; ++t)
                    if (ok[t] && ncq[t] >= CHUNK_IDS)
                        ok[t] = write_chunk(ws.cq + t * CQ_TILE, CHUNK_IDS, ncq[t], head[t], count[t]);
            }
        }
#pragma unroll
        for (int t = 0; t < TILES_PER_GROUP; ++t) {
            if (!valid[t]) continue;
            if (ok[t] && ncq[t] > 0) ok[t] = write_chunk(ws.cq + t * CQ_TILE, ncq[t], ncq[t], head[t], count[t]);
            finish_tile(group * TILES_PER_GROUP + t, head[t], count[t], ok[t]);
        }
    } else if (P.heavy_slab) {
        // ---- the group's list did not fit shared memory: k_heavy_lists (next on the stream) lists it in depth slabs
        // and writes the four descriptors (heavy_lists.cuh)
        if (lane == 0) P.heavy_groups[atomicAdd(P.counters + CTR_HEAVY, 1u)] = group;
    } else if (P.heavy_fused) {
        // ---- the group's list did not fit shared memory: its frustum holds ~1000 Gaussians or more, typically
        // because it looks along a surface.  Listing them all is the wrong plan - the rays will have their K
        // nearest hits after a small part of them - so the tiles go to the fused kernel, which traverses near
        // first and prunes by distance as its hit buffers fill (fused.cuh)
#pragma unroll 1
        for (int sub = 0; sub < TILES_PER_GROUP; ++sub) {
            const int i0 = gi0 + (sub / GROUP_TJ) * TILE_I, j0 = gj0 + (sub % GROUP_TJ) * TILE_J;
            if (i0 >= xe || j0 >= ye) continue;
            finish_tile(group * TILES_PER_GROUP + sub, -1, 0, false);
        }
        // tell the host that this scene has heavy groups: later frames run k_heavy_lists for them (render.cu)
        if (lane == 0 && !S.heavy_flagged) {
            *reinterpret_cast<volatile int*>(P.mirror + 2) = 1;
            S.heavy_flagged = true;
        }
    } else {
        // ---- (RTGS_HEAVY_FUSED=0) one traversal per tile, leaves stream out -------
#pragma unroll 1
        for (int sub = 0; sub < TILES_PER_GROUP; ++sub) {
            const int i0 = gi0 + (sub / GROUP_TJ) * TILE_I, j0 = gj0 + (sub % GROUP_TJ) * TILE_J;
            if (i0 >= xe || j0 >= ye) continue;
            Frustum fr;
            make_frustum(cam, i0, i0 + TILE_I, j0, j0 + TILE_J, fr);
            int head = -1, count = 0, ncq = 0;
            bool ok = true;
            int top = 1;
            if (lane == 0) ws.glist[0] = 0;
            __syncwarp();
#pragma unroll 1
            while (top > 0 && ok) {
                traverse_step(ws.glist, top, ws.cq, ncq, fr);
                ST(S.st_max_stack = max(S.st_max_stack, (unsigned)top));
#pragma unroll 1
                while (ncq >= CHUNK_IDS && ok) ok = write_chunk(ws.cq, CHUNK_IDS, ncq, head, count);
            }
            if (ok && ncq > 0) ok = write_chunk(ws.cq, ncq, ncq, head, count);
            finish_tile(group * TILES_PER_GROUP + sub, head, count, ok);
            __syncwarp();
        }
    }
    // ---- publish: descriptors and chunks of this group are complete (lane 0 wrote the descriptors, every lane
    // wrote chunk words; __syncwarp orders them before lane 0's release, which is cumulative)
    if (P.ready != nullptr) {   // (separate launches: the kernel boundary publishes everything)
        __syncwarp();
        if (lane == 0)
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(P.ready + group), "r"(P.seq) : "memory");
    }
#undef ST
}

}  // namespace rtgs_dev
