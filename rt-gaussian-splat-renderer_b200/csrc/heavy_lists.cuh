// heavy_lists.cuh — depth-capped candidate lists for the tiles of HEAVY groups: 8x16-pixel groups whose frustum holds
// more Gaussians than the shared-memory list of tile_lists.cuh (typically because they look along a surface: thousands
// of splats, of which every ray composites the nearest 16, ray_tracer.py:96-104).  Listing them all is the wrong plan,
// and the fused kernel's near-first traversal with a sorted stack (fused.cuh) costs ~77 k warp instructions per tile.
// Here a warp walks ONE 4x8-pixel tile of such a group in DEPTH SLABS:
//
//   depth z(box) = min over the box of (x - o).c / L,  c = unit direction of the tile's centre ray, L >= |d| of every
//   ray of the tile: a lower bound of the ray parameter t of any point of the box on any ray of the tile.
//
//   1. traverse the tile's frustum with a cap: children with z < cap are expanded / listed as in lists_group,
//      children with z >= cap are DEFERRED (appended, with their depth, to a per-warp list in global memory);
//   2. the new candidates are filtered (exact ellipsoid-vs-frustum test) and run through the SAME hit test as the
//      shading (stage_candidate / coarse mask / precise_test of render_common.cuh, lane = pixel); every ray keeps the
//      entry distances of its 16 nearest hits;
//   3. while some ray holds fewer than 16 hits, or its 16th hit lies behind the nearest deferred depth, the cap is
//      raised and the deferred list re-scanned.  The new cap is a rank statistic of the deferred depths (the
//      SLAB_RANK-th smallest of the 32 lanes' nearest deferred depths), so a pass activates a few dozen entries
//      whatever the local density: no steps through empty space, no plunge into a surface; a pass that overflows
//      the shared list is repeated with a nearer cap.
//
// The walk ends when the farthest 16th hit of the tile lies in front of everything deferred.  The candidates nearer than
// that limit are published as the tile's list together with the limit (TileDesc::count | TILE_CAPPED, tile_cap[tile]):
// everything that can enter a ray of the tile nearer than the limit is in the list by construction.  The shading
// re-derives the hits from the list and checks the claim - a tile is decided iff every ray holds K hits nearer than the
// limit (shade.cuh) - so nothing depends on this file being right about the hits, only the speed does; a tile that is
// not decided, or whose slab overflows, goes to the fused kernel as before.
//
// OPT-IN (RTGS_OPT_HEAVY_LISTS), measured on the surface-like scene (1 M Gaussians, 1080p, 12 % of the tiles in heavy
// groups, DESIGN.md §8): every heavy tile is decided by its slab (0-30 of ~8000 fail, 1-2 go to the fused kernel), the
// frames are bit-identical, 180-220 candidates are tested per tile against the 511 the fused kernel stages - but the
// walk costs 8-9 passes and ~380 k cycles per tile on 16 warps per SM (40 % of it the hit tests, the rest dependent
// node and list fetches), 1.0 ms per frame against the 1.37 ms of k_render it replaces, and the shading gains 0.17 ms
// for the longer lists: 2.48 vs 2.36 ms per frame, 1141 vs 1134 Mrays/s for the two-stream sweep.  No gain, so the
// default stays the fused kernel.
#pragma once
#include "shade.cuh"
#include "tile_lists.cuh"

namespace rtgs_dev {

constexpr int HEAVY_K = 16;              // hits a ray keeps (the k-buffer depth of the shading)
constexpr int HEAVY_MAX_ITERS = 128;     // passes per tile before it is handed to the fused kernel
constexpr int HEAVY_LIST_LIMIT = GLIST_CAP - 4 * LISTS_TAKE;
constexpr float HEAVY_MARGIN = 1.0001f;  // limit = farthest 16th hit x this (float32 rounding of depths and distances)
// The cap of a pass is the SLAB_RANK-th smallest of the 32 lanes' nearest deferred depths (surface-like scene, heavy
// lists from the first frame: 2.48 ms per frame at 24, 2.54 ms at 16; profiles/r02_heavy_lists_probe.log).
constexpr int SLAB_RANK = 24;

struct __align__(16) HeavyShared {
    ListsShared l;                         // traversal stack, the tile's candidates so far, output queue
    StagedRecords rec;                     // staging of one batch of candidates (as ShadeShared)
    float4 polyA[SHADE_BATCH];
    float2 polyB[SHADE_BATCH];
};

struct HeavyStats {
    unsigned long long tiles = 0, failed = 0, iters = 0, tested = 0, retries = 0, fail_list = 0, fail_defer = 0,
                       fail_passes = 0;
    unsigned max_deferred = 0;
    unsigned long long cyc_walk = 0, cyc_test = 0, cyc_publish = 0;   // SM clock cycles per phase (statistics builds)
};

// One tile of a heavy group.  `def` = this warp's deferred lists: 2 x P.heavy_defer_cap entries {child id (< 0: ~leaf),
// depth bits}; `hint` = a first guess of the limit (0: none).  Returns the guess for a neighbouring tile.  (The kernel
// passes no hints: walking the four tiles of a group one after the other with the neighbour's limit as first cap saves a
// third of the cycles per tile, 304 k against 383-490 k, but leaves a quarter of the work items - 1.3 ms instead of 1.0.)
template <bool STATS>
__device__ __noinline__ float heavy_tile(const RenderParams& P, HeavyShared& hs, ListsState& S, HeavyStats& HS,
                                         int2* __restrict__ def, int tile, int i0, int j0, float hint, int lane) {
    ListsShared& ws = hs.l;
    const unsigned lt_mask = (1u << lane) - 1u;
    const CamD& cam = P.cam;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
    const int dcap = P.heavy_defer_cap;
#define ST(expr) do { if (STATS) { expr; } } while (0)

    const long long t_begin = STATS ? clock64() : 0;
    const int pi = i0 + lane / TILE_J, pj = j0 + lane % TILE_J;
    const bool active = pi < xe && pj < ye;
    TileRays tr;
    make_tile_rays(cam, i0, j0, pi, pj, active, tr);
    Frustum ft;
    make_frustum(cam, i0, min(i0 + TILE_I, xe), j0, min(j0 + TILE_J, ye), ft);

    // ---- the depth functional --------------------------------------------------------------------------------------
    float zc[3], za[3], zo;
    {
        const d3 dc = cam_dir(cam, (double)i0 + 0.5 * TILE_I, (double)j0 + 0.5 * TILE_J);   // tile-centre ray
        // L: the longest direction among the tile's corner and centre rays (1 for a unit camera quaternion), plus a
        // margin for the rays in between
        double l2 = d3dot(dc, dc);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const d3 e = cam_dir(cam, (double)(i0 + (k & 1) * TILE_I), (double)(j0 + (k >> 1) * TILE_J));
            l2 = fmax(l2, d3dot(e, e));
        }
        const double sc = 1.0 / (sqrt(d3dot(dc, dc)) * sqrt(l2) * 1.0001);
        zc[0] = (float)(dc.x * sc); zc[1] = (float)(dc.y * sc); zc[2] = (float)(dc.z * sc);
#pragma unroll
        for (int k = 0; k < 3; ++k) za[k] = fabsf(zc[k]);
        zo = zc[0] * (float)cam.o[0] + zc[1] * (float)cam.o[1] + zc[2] * (float)cam.o[2];
    }
    auto box_depth = [&](float cx, float cy, float cz, float hx, float hy, float hz) {
        return zc[0] * cx + zc[1] * cy + zc[2] * cz - za[0] * hx - za[1] * hy - za[2] * hz - zo;
    };

    // ---- per ray: entry distances of the nearest HEAVY_K hits (unordered), the farthest of them ----------------------
    float kb[HEAVY_K];
    int kcnt = 0, kslot = 0;
    float kmax = INFINITY;   // the HEAVY_K-th nearest entry distance once kcnt == HEAVY_K

    int nk = 0;              // glist[0, nk): candidates that passed the ellipsoid filter and have been tested
    int ng = 0;              // glist[nk, ng): leaves found since
    int top = 0;
    bool failed = false;
    int why = 0;   // 1 = the slab overflowed the shared list, 2 = the deferred list overflowed, 3 = too many passes
    int n_in = 0, n_out = 0;
    int2* din = def;
    int2* dout = def + dcap;
    float zmin = INFINITY;   // per lane: nearest depth among the entries this lane deferred in this pass

    // expand what is on the stack, depth first, against `cap` (traverse_step of tile_lists.cuh plus the depth test)
    auto drain = [&](float cap, float cap_leaf) {
#pragma unroll 1
        while (top > 0 && !failed) {
            const int take = top > P.lists_single ? 1 : min(16, top);
            int node = -1;
            if ((lane >> 1) < take) node = ws.stack[top - 1 - (lane >> 1)];
            top -= take;
            __syncwarp();
            bool h0 = false, h1 = false;
            int c0 = 0, c1 = 0;
            float z0 = 0.0f, z1 = 0.0f;
            if (node >= 0) {
                const float4* rec = P.nodes4 + (int64_t)node * 8 + (lane & 1) * 4;
                float4 a, b, c, d;
                ldg256(rec + 0, a, b);
                ldg256(rec + 2, c, d);
                c0 = __float_as_int(d.x);
                c1 = __float_as_int(d.y);
                h0 = box_in_frustum(ft, a.x, a.y, a.z, a.w, b.x, b.y);
                h1 = box_in_frustum(ft, b.z, b.w, c.x, c.y, c.z, c.w);
                z0 = box_depth(a.x, a.y, a.z, a.w, b.x, b.y);
                z1 = box_depth(b.z, b.w, c.x, c.y, c.z, c.w);
            }
            ST(S.st_nodes += 4ull * (unsigned)take);
            ST(S.st_steps += 1);
            // near: expand (internal nodes below the traversal cap) / list now (leaves below the test cap)
            const bool n0 = h0 && z0 < (c0 >= 0 ? cap : cap_leaf), n1 = h1 && z1 < (c1 >= 0 ? cap : cap_leaf);
            const bool f0 = h0 && !n0, f1 = h1 && !n1;             // far: deferred
            const unsigned mI0 = __ballot_sync(FULL, n0 && c0 >= 0), mI1 = __ballot_sync(FULL, n1 && c1 >= 0);
            const unsigned mL0 = __ballot_sync(FULL, n0 && c0 < 0), mL1 = __ballot_sync(FULL, n1 && c1 < 0);
            const unsigned mF0 = __ballot_sync(FULL, f0), mF1 = __ballot_sync(FULL, f1);
            if (n0 && c0 >= 0) ws.stack[top + __popc(mI0 & lt_mask)] = c0;
            const int topa = top + __popc(mI0);
            if (n1 && c1 >= 0) ws.stack[topa + __popc(mI1 & lt_mask)] = c1;
            top = topa + __popc(mI1);
            if (ng + __popc(mL0) + __popc(mL1) > HEAVY_LIST_LIMIT || n_out + __popc(mF0) + __popc(mF1) > dcap) {
                failed = true;   // the slab itself overflows the shared list (or the deferred list): fused kernel
                why = ng + __popc(mL0) + __popc(mL1) > HEAVY_LIST_LIMIT ? 1 : 2;
                break;
            }
            if (n0 && c0 < 0) ws.glist[ng + __popc(mL0 & lt_mask)] = ~c0;
            const int nga = ng + __popc(mL0);
            if (n1 && c1 < 0) ws.glist[nga + __popc(mL1 & lt_mask)] = ~c1;
            ng = nga + __popc(mL1);
            if (f0) {
                dout[n_out + __popc(mF0 & lt_mask)] = make_int2(c0, __float_as_int(z0));
                zmin = fminf(zmin, z0);
            }
            const int noa = n_out + __popc(mF0);
            if (f1) {
                dout[noa + __popc(mF1 & lt_mask)] = make_int2(c1, __float_as_int(z1));
                zmin = fminf(zmin, z1);
            }
            n_out = noa + __popc(mF1);
            __syncwarp();
            ST(S.st_max_stack = max(S.st_max_stack, (unsigned)top));
        }
    };

    // The leaves found since the last call, glist[nk, ng): exact ellipsoid-vs-frustum filter, the survivors compacted in
    // place behind glist[0, nk) and run through the shading's hit test, 32 at a time (shade.cuh: stage, coarse, precise)
    auto test_new = [&]() {
#pragma unroll 1
        for (int base = nk; base < ng; base += 32) {
            const int idx = base + lane;
            int s = 0;
            bool keep = false;
            if (idx < ng) {
                s = ws.glist[idx];
                float4 a, b;
                ldg256(P.leafbox + (int64_t)s * 2, a, b);
                keep = ellipsoid_in_frustum(ft, a, b);
            }
            const unsigned mk = __ballot_sync(FULL, keep);
            const int m = __popc(mk);
            __syncwarp();   // every lane has read its entry: the compaction may overwrite the batch
            if (keep) ws.glist[nk + __popc(mk & lt_mask)] = s;
            __syncwarp();
            const int m4 = (m + 3) & ~3;
            if (lane < m) {
                float4 rec[REC_QUADS];
                float poly[6], t_lo;
                stage_candidate(P, tr, ws.glist[nk + lane], rec, poly, t_lo);
#pragma unroll
                for (int k = 0; k < REC_QUADS; ++k) hs.rec[k][lane] = rec[k];
                hs.polyA[lane] = make_float4(poly[0], poly[1], poly[2], poly[3]);
                hs.polyB[lane] = make_float2(poly[4], poly[5]);
            } else if (lane < m4) {
                hs.polyA[lane] = make_float4(1.0f, 0.0f, 0.0f, 0.0f);
                hs.polyB[lane] = make_float2(0.0f, 0.0f);
            }
            __syncwarp();
            unsigned mask = 0;
#pragma unroll 1
            for (int c = 0; c < m4; c += 4) {
                unsigned nib = 0;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float4 pA = hs.polyA[c + u];
                    const float2 pB = hs.polyB[c + u];
                    const float ta = fmaf(tr.pa, pA.w, fmaf(tr.pb, pB.x, pA.y));
                    const float tb = fmaf(tr.pb, pB.y, pA.z);
                    const float Sq = fmaf(tr.pa, ta, fmaf(tr.pb, tb, pA.x));
                    if (Sq < 0.0f) nib |= 1u << u;
                }
                mask |= nib << c;
            }
            if (!active) mask = 0;
#pragma unroll 1
            while (__any_sync(FULL, mask != 0)) {
                if (mask != 0) {
                    const int c = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const PreciseHit h = precise_test(P, hs.rec, c, tr, pi, pj);
                    if (h.hit && h.t1 < kmax) {
                        const int slot = kcnt < HEAVY_K ? kcnt : kslot;
                        kb[slot] = h.t1;
                        if (kcnt < HEAVY_K) ++kcnt;
                        if (kcnt == HEAVY_K) {
                            float mt = -INFINITY;
#pragma unroll
                            for (int k = 0; k < HEAVY_K; ++k)
                                if (kb[k] > mt) { mt = kb[k]; kslot = k; }
                            kmax = mt;
                        }
                    }
                }
            }
            __syncwarp();
            nk += m;
            ST(HS.tested += (unsigned)m);
        }
        ng = nk;
    };

    // ---- the slab walk -------------------------------------------------------------------------------------------
    // pass 0: the root is expanded unconditionally with cap = -inf, i.e. its grandchildren are all deferred
    if (lane == 0) ws.stack[0] = 0;
    top = 1;
    __syncwarp();
    drain(-INFINITY, -INFINITY);
    // The cap of a pass comes from the depths of what is deferred: every lane remembers the nearest depth among the
    // entries it deferred itself (entries are spread over the lanes as they come), and the cap is the SLAB_RANK-th
    // smallest of those 32 values - so a pass activates a few dozen entries whatever the local density is: no steps
    // through empty space, no plunge into a surface.  The first pass of a tile whose neighbour has just been walked
    // goes straight to that tile's limit (`hint`).
    float limit = INFINITY;
    int iters = 0;
    int pending = 0;         // leaves in glist[nk, ng) that have not been tested yet
    bool full = false;       // every ray holds HEAVY_K hits
    float want = INFINITY;   // the farthest HEAVY_K-th hit x HEAVY_MARGIN
#pragma unroll 1
    while (!failed) {
        // what the pass deferred: count n_out, nearest depth zm, SLAB_RANK-th of the lanes' nearest depths zr
        ST(HS.max_deferred = max(HS.max_deferred, (unsigned)n_out));
        float zs = zmin;
#pragma unroll
        for (int k = 2; k <= 32; k <<= 1) {      // bitonic sort of the 32 lane values, ascending by lane
#pragma unroll
            for (int j = k >> 1; j > 0; j >>= 1) {
                const float o = __shfl_xor_sync(FULL, zs, j);
                const bool up = ((lane & k) == 0) == ((lane & j) == 0);
                zs = up ? fminf(zs, o) : fmaxf(zs, o);
            }
        }
        const float zm = __shfl_sync(FULL, zs, 0);
        float zr = __shfl_sync(FULL, zs, SLAB_RANK);
        if (!(zr < INFINITY)) {                  // fewer lanes than that hold entries: the farthest of them
            float f = zs < INFINITY ? zs : -INFINITY;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) f = fmaxf(f, __shfl_xor_sync(FULL, f, o));
            zr = f;
        }
        pending = ng - nk;
        // the hit test works on batches of 32: while some ray is short of hits anyway, a handful of new leaves waits
        // for the next pass
        if (pending > 0 && (full || pending >= 24 || n_out == 0)) {
            const long long t0 = STATS ? clock64() : 0;
            test_new();
            ST(HS.cyc_test += (unsigned long long)(clock64() - t0));
            pending = 0;
            full = __all_sync(FULL, !active || kcnt == HEAVY_K);
            float est = active ? kmax : 0.0f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) est = fmaxf(est, __shfl_xor_sync(FULL, est, o));
            want = est * HEAVY_MARGIN;
        }
        if (n_out == 0) {                // nothing deferred: the list is the tile's whole frustum
            limit = full ? want : INFINITY;
            break;
        }
        if (full && want <= zm) {        // nothing nearer than the wanted limit is deferred
            limit = want;
            break;
        }
        // the deferred list of the last pass becomes the input of this one; a pass that overflows the shared list is
        // repeated with a cap nearer to zm (its input is untouched)
        { int2* t = din; din = dout; dout = t; }
        n_in = n_out;
        float reach = 1.0f;
#pragma unroll 1
        for (;;) {
            if (++iters > HEAVY_MAX_ITERS) {
                failed = true;
                why = 3;
                break;
            }
            float cap = zm + (zr - zm) * reach;
            cap = fmaxf(cap * 1.000001f, zm > 0.0f ? zm * 1.002f : 1e-30f);
            if (iters == 1 && hint > cap) cap = hint;
            // never beyond what the rays ask for (their 16th hits so far may lie far behind the slab - a huge blob
            // whose box begins in it - and move in as nearer candidates are found)
            const bool last = full && want * 1.000001f <= cap;
            if (last) cap = want * 1.000001f;
            ng = nk + pending;
            n_out = 0;
            top = 0;
            zmin = INFINITY;
            failed = false;
            __syncwarp();
            // entries below the cap are expanded (internal nodes) or listed (leaves), the rest is deferred again; the
            // next batch is in flight while this one is handled
            int2 e_next = make_int2(0, 0);
            if (lane < n_in) e_next = __ldcg(din + lane);
#pragma unroll 1
            for (int base = 0; base < n_in && !failed; base += 32) {
                const int2 e = e_next;
                const bool have = base + lane < n_in;
                if (base + 32 + lane < n_in) e_next = __ldcg(din + base + 32 + lane);
                const float z = __int_as_float(e.y);
                const bool nearb = have && z < cap;
                const bool farb = have && !nearb;
                const unsigned mI = __ballot_sync(FULL, nearb && e.x >= 0), mL = __ballot_sync(FULL, nearb && e.x < 0),
                               mF = __ballot_sync(FULL, farb);
                if (ng + __popc(mL) > HEAVY_LIST_LIMIT || n_out + __popc(mF) > dcap) {
                    failed = true;
                    why = ng + __popc(mL) > HEAVY_LIST_LIMIT ? 1 : 2;
                    break;
                }
                if (nearb && e.x >= 0) ws.stack[top + __popc(mI & lt_mask)] = e.x;
                top += __popc(mI);
                if (nearb && e.x < 0) ws.glist[ng + __popc(mL & lt_mask)] = ~e.x;
                ng += __popc(mL);
                if (farb) {
                    dout[n_out + __popc(mF & lt_mask)] = e;
                    zmin = fminf(zmin, z);
                }
                n_out += __popc(mF);
                __syncwarp();
                // the activated nodes collect on the stack and are expanded 16 at a time; above the batch threshold
                // (<= 32 entries over it here: within the bound of tile_lists.cuh) the stack is drained first
                if (top > P.lists_single) drain(cap, cap);
            }
            if (!failed) drain(cap, cap);
            if (!failed) break;
            if (why != 1 || last || reach < 0.01f) break;
            reach *= 0.25f;
            hint = 0.0f;
            ST(HS.retries += 1);
        }
    }
    ST(HS.iters += (unsigned)iters);
    ST(HS.tiles += 1);
    const long long t_walk_end = STATS ? clock64() : 0;
    ST(HS.cyc_walk += (unsigned long long)(t_walk_end - t_begin));
    ST(S.st_max_list = max(S.st_max_list, (unsigned)ng));

    if (failed) {
        ST(HS.failed += 1);
        ST(HS.fail_list += why == 1);
        ST(HS.fail_defer += why == 2);
        ST(HS.fail_passes += why == 3);
        if (lane == 0) {
            atomicAdd(P.counters + CTR_HEAVY_FAILED, 1u);
            TileDesc d;
            d.head = -1;
            d.count = -1;
            P.desc[tile] = d;
            P.fallback_tiles[atomicAdd(P.counters + CTR_FALLBACK, 1u)] = tile;
        }
        return 0.0f;
    }

    // ---- publish glist[0, nk) nearer than the limit, in pool chunks (as in lists_group) ---------------------------
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
    int head = -1, count = 0, ncq = 0;
    bool ok = true;
    auto write_chunk = [&](int m) {
        const int chunk = alloc_chunk();
        if (chunk < 0) {
            ok = false;
            return;
        }
        int v = head;
        if (lane < m) v = ws.cq[ncq - m + lane];
        if (lane < m || lane == CHUNK_INTS - 1) P.pool[(int64_t)chunk * CHUNK_INTS + lane] = v;
        head = chunk;
        ncq -= m;
        count += m;
        __syncwarp();
    };
#pragma unroll 1
    for (int base = 0; base < nk && ok; base += 32) {
        const int idx = base + lane;
        int s = 0;
        bool keep = false;
        if (idx < nk) {
            s = ws.glist[idx];
            float4 a, b;
            ldg256(P.leafbox + (int64_t)s * 2, a, b);
            keep = box_depth(a.x, a.y, a.z, a.w, b.x, b.y) < limit;
        }
        const unsigned mk = __ballot_sync(FULL, keep);
        if (keep) ws.cq[ncq + __popc(mk & lt_mask)] = s;
        ncq += __popc(mk);
        __syncwarp();
        while (ok && ncq >= CHUNK_IDS) write_chunk(CHUNK_IDS);
    }
    if (ok && ncq > 0) write_chunk(ncq);
    if (lane == 0) {
        TileDesc d;
        d.head = head;
        d.count = !ok ? -1 : (limit < INFINITY ? (count | TILE_CAPPED) : count);
        P.desc[tile] = d;
        // (1 - 1e-5: depths and distances are float32 values; the shading requires kmax < this)
        if (ok && limit < INFINITY) P.tile_cap[tile] = limit * (1.0f - 1e-5f);
        if (!ok) P.fallback_tiles[atomicAdd(P.counters + CTR_FALLBACK, 1u)] = tile;
    }
    ST(S.st_cands += ok ? (unsigned)count : 0u);
    ST(HS.cyc_publish += (unsigned long long)(clock64() - t_walk_end));
#undef ST
    return limit < INFINITY ? limit * 0.98f : 0.0f;   // the neighbouring tile's first guess
}

}  // namespace rtgs_dev
