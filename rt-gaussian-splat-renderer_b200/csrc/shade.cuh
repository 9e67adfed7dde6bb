// shade.cuh — everything of the render path after the traversal, per 4x8-pixel tile (device code shared by the
// stand-alone k_shade_tiles kernel and the single-launch frame kernel k_frame, render.cu):
//   camera ray generation        camera.py:31-71              (registers; rays never stored)
//   ray-Gaussian intersection    gaussian.py:203-230          (local-frame quadratic)
//   response + SH colour         gaussian.py:140-201
//   front-to-back compositing    ray_tracer.py:79-104         (k-buffer of the `depth` nearest entries)
//
// A warp owns one tile at a time (lane = pixel) and walks the tile's candidate list, 31 candidates (one
// 128-byte chunk) per batch:
//   stage    one lane per candidate, float64: origin shifted to the closest point of the tile's centre
//            ray -> a 64-byte float32 record in the camera's pixel basis + a 6-coefficient quadratic in shared
//            memory;
//   coarse   every lane evaluates every staged quadratic (broadcast shared-memory reads, 5 FMA) and
//            keeps a 32-bit mask of the candidates its ray may hit;
//   precise  warp-wide rounds, each lane takes the next set bit of its mask: exact decision (float32
//            linear in the pixel offset, float64 from the raw parameters inside the error band), entry
//            distance, alpha; the hit goes to the lane's K-entry buffer in shared memory (replace-max
//            once K are held; the nearest hit left outside is remembered, and if it is within float32
//            rounding of the farthest kept entry the two are compared in float64 after the list).
// After the list: the lane's entries are ordered by a bitonic network over (entry-distance bits | slot) keys in
// registers (near ties by their float64 entry distances), composited in that order with the SH basis evaluated
// once per ray (six 256-bit loads per layer), and stored sector-aligned.
//
// Numerics: identical to the fused kernel (fused.cuh) - parity is defined against the float64
// evaluation of the reference's maths, see DESIGN.md §2.
//
// The code is bound by the L1 data pipe (per-lane gathers of SH and staged records), not by latency:
// 20 warps x 96 registers per SM is the measured optimum, 9.0 KB of shared memory per warp (9232 bytes).
#pragma once
#include "kbuffer.cuh"

namespace rtgs_dev {

constexpr int SHADE_K = 16;          // k-buffer entries (depth <= 16)
constexpr float TIE_BAND = 2e-6f;    // relative: float32 entry distances closer than this are compared in float64
constexpr int SHADE_BATCH = REC_BATCH;   // staged candidates per batch (a chunk fills 31)

struct __align__(16) ShadeShared {
    StagedRecords rec;                     // precise records; the output staging of store_tile
    float4 polyA[SHADE_BATCH];             // coarse quadratics {c0 c1 c2 c3}
    float2 polyB[SHADE_BATCH];             //                   {c4 c5}
    float kb_t[SHADE_K][32];               // per-lane hit buffer (unsorted): entry distance, sorted position, alpha
    int kb_i[SHADE_K][32];
    float kb_a[SHADE_K][32];
    float amb[2][32];                      // per lane: id and alpha of the nearest hit that is NOT in the buffer
    int band_state[4];                     // lane 0's band-completion counts (render_common.cuh: BandCount)
};

struct ShadeStats {
    unsigned long long st_useful = 0, st_pairs = 0, st_f64 = 0, st_layers = 0, st_hit = 0, st_rays = 0, st_tiles = 0,
                       st_ins = 0;
};

// Shade tile `tile` (a valid id < P.ntiles whose descriptor has been published).  DEPTH: also the composited ray
// distance (render_common.cuh: composite_depth) to P.out_depth.
template <bool STATS, bool DEPTH = false>
__device__ __forceinline__ void shade_tile(const RenderParams& P, ShadeShared& ws, ShadeStats& S, PeerGrant& G,
                                           BandCount& BC, int tile, int lane) {
    constexpr int K = SHADE_K;
    constexpr int BATCH = SHADE_BATCH;
    const CamD& cam = P.cam;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
#define ST(expr) do { if (STATS) { expr; } } while (0)
    int i0, j0;
    tile_origin(P, tile, i0, j0);
    const TileDesc desc = load_desc(P, tile);
    if (desc.count < 0) return;   // list did not fit the pool: the fused kernel renders this tile
    const bool capped = (desc.count & TILE_CAPPED) != 0;   // depth-capped list of a heavy group (heavy_lists.cuh)
    const int desc_count = desc.count & ~TILE_CAPPED;
    const int pi = i0 + lane / TILE_J, pj = j0 + lane % TILE_J;
    const bool active = pi < xe && pj < ye;

    int cnt = 0;
    // The K nearest hits are kept by their float32 entry distances (replace-max once the buffer is full).  Which
    // of two hits is nearer is only certain beyond float32 rounding (TIE_BAND), so the one place where it
    // matters - the boundary between the K-th and the (K+1)-th nearest - is re-examined in float64 after the
    // list: e1_t / ws.amb hold the nearest hit that is NOT in the buffer (a rejected hit or an evicted entry),
    // bit 8 of kmax_slot says that a second such hit lies within float32 rounding of it.  (Checking every
    // transient boundary instead sent 8 % of the dense tiles of a surface-like scene to the fused kernel:
    // a ray with 1000 hits replaces its farthest entry ~60 times.)
    float e1_t = INFINITY, kmax_t = INFINITY;
    int kmax_slot = 0;
    TileRays tr;
    if (desc_count > 0) {
        make_tile_rays(cam, i0, j0, pi, pj, active, tr);
        int left = desc_count;
        // one coalesced 128-byte read per chunk: lanes 0..30 candidates, lane 31 the next chunk (L2 only: in k_frame
        // the chunks are written by other warps of the same launch)
        int cur = __ldcg(P.pool + (int64_t)desc.head * CHUNK_INTS + lane);
#pragma unroll 1
        while (left > 0) {
            const int m = (left - 1) % CHUNK_IDS + 1;
            left -= m;
            const int s = cur;
            const int next = __shfl_sync(FULL, cur, CHUNK_INTS - 1);
            if (left > 0) cur = __ldcg(P.pool + (int64_t)next * CHUNK_INTS + lane);   // prefetch
            // ---- stage ---------------------------------------------------------------------
            const int m4 = (m + 3) & ~3;
            if (lane < m) {
                float4 rec[REC_QUADS];
                float poly[6], t_lo;
                stage_candidate(P, tr, s, rec, poly, t_lo);
#pragma unroll
                for (int k = 0; k < REC_QUADS; ++k) ws.rec[k][lane] = rec[k];
                ws.polyA[lane] = make_float4(poly[0], poly[1], poly[2], poly[3]);
                ws.polyB[lane] = make_float2(poly[4], poly[5]);
            } else if (lane < m4) {   // pad to a multiple of 4: never a candidate
                ws.polyA[lane] = make_float4(1.0f, 0.0f, 0.0f, 0.0f);
                ws.polyB[lane] = make_float2(0.0f, 0.0f);
            }
            __syncwarp();
            ST(S.st_pairs += (unsigned)m);
            // ---- coarse: mask of the staged candidates this ray may hit ---------------------
            unsigned mask = 0;
#pragma unroll 1
            for (int c = 0; c < m4; c += 4) {
                unsigned nib = 0;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float4 pA = ws.polyA[c + u];
                    const float2 pB = ws.polyB[c + u];
                    const float ta = fmaf(tr.pa, pA.w, fmaf(tr.pb, pB.x, pA.y));   // c1 + a c3 + b c4
                    const float tb = fmaf(tr.pb, pB.y, pA.z);                      // c2 + b c5
                    const float S = fmaf(tr.pa, ta, fmaf(tr.pb, tb, pA.x));
                    if (S < 0.0f) nib |= 1u << u;
                }
                mask |= nib << c;
            }
            if (!active) mask = 0;
            ST(S.st_useful += (unsigned)__popc(__reduce_or_sync(FULL, mask)));
            // ---- precise: warp-wide rounds, one candidate per lane and round -----------------
#pragma unroll 1
            while (__any_sync(FULL, mask != 0)) {
                if (mask != 0) {
                    const int c = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const PreciseHit h = precise_test(P, ws.rec, c, tr, pi, pj);
                    ST(S.st_f64 += h.refined);
                    if (h.hit) {
                        float xt = h.t1, xa = h.alpha;   // the hit that stays outside the buffer (full buffer)
                        int xi = h.s;
                        int slot = -1;
                        if (cnt < K) {
                            slot = cnt++;
                        } else if (h.t1 < kmax_t) {   // full: replace the farthest entry, which goes outside
                            slot = kmax_slot & 15;
                            xt = kmax_t;
                            xi = ws.kb_i[slot][lane];
                            xa = ws.kb_a[slot][lane];
                        }
                        const bool full = cnt == K;
                        if (slot >= 0) {
                            ws.kb_t[slot][lane] = h.t1;
                            ws.kb_i[slot][lane] = h.s;
                            ws.kb_a[slot][lane] = h.alpha;
                            if (full) {   // track the farthest entry (exact float32 maximum)
                                float mt = -INFINITY;
                                int ms = 0;
#pragma unroll
                                for (int k = 0; k < K; ++k) {
                                    const float t = ws.kb_t[k][lane];
                                    if (t > mt) { mt = t; ms = k; }
                                }
                                kmax_slot = ms | (kmax_slot & 0x100);
                                if (kmax_t == INFINITY) xt = INFINITY;   // the buffer has just filled: nothing is outside yet
                                kmax_t = mt;
                            }
                        }
                        if (full && xt < INFINITY) {
                            if (xt < e1_t) {
                                kmax_slot = (e1_t - xt <= TIE_BAND * xt) ? (kmax_slot | 0x100) : (kmax_slot & ~0x100);
                                e1_t = xt;
                                ws.amb[0][lane] = __int_as_float(xi);
                                ws.amb[1][lane] = xa;
                            } else if (xt - e1_t <= TIE_BAND * e1_t) {
                                kmax_slot |= 0x100;
                            }
                        }
                    }
                }
                ST(S.st_ins += 1);
            }
            __syncwarp();
        }
    }

    // ---- a depth-capped list holds every Gaussian that can enter a ray of the tile nearer than tile_cap[tile]: the
    // tile is decided iff every ray has its K hits nearer than that (the cap is a guess from sample rays); if not,
    // k_render renders the tile from scratch, as for the near-ties below
    if (capped) {
        const float cap = __ldcg(P.tile_cap + tile);
        if (__any_sync(FULL, active && !(cnt == K && kmax_t < cap))) {
            if (lane == 0) {
                P.fallback_tiles2[atomicAdd(P.counters + CTR_FALLBACK2, 1u)] = tile;
                *reinterpret_cast<volatile int*>(P.mirror + 1) = 1;
            }
            return;
        }
    }

    // ---- the K-th / (K+1)-th boundary (rare): is the nearest outside hit within float32 rounding of the
    // farthest entry?  Then their float64 entry distances decide, repeatedly while the loser ties again.
    const bool amb = e1_t - kmax_t <= TIE_BAND * kmax_t;   // false while either is inf
    if (__any_sync(FULL, amb)) {
        if (__any_sync(FULL, amb && (kmax_slot & 0x100))) {
            // three contenders within rounding: k_render (launched next on the stream) renders the tile and
            // resolves them on the spot; nothing of it has been written yet, so `accumulate` outputs stay correct
            if (lane == 0) {
                P.fallback_tiles2[atomicAdd(P.counters + CTR_FALLBACK2, 1u)] = tile;
                *reinterpret_cast<volatile int*>(P.mirror + 1) = 1;
            }
            return;
        }
        if (amb) {
            float ct = e1_t, ca = ws.amb[1][lane];
            int ci = __float_as_int(ws.amb[0][lane]);
            float mt = kmax_t;
            int ms = kmax_slot & 15;
#pragma unroll 1
            for (int it = 0; it < 4; ++it) {
                if (!(ct - mt <= TIE_BAND * mt)) break;
                ST(S.st_f64 += 2);
                if (!exact_less(P.raw, cam, ci, ws.kb_i[ms][lane], pi, pj)) break;
                // the outside hit is nearer: it takes the slot, the former farthest entry is the contender now
                const float ot = mt, oa = ws.kb_a[ms][lane];
                const int oi = ws.kb_i[ms][lane];
                ws.kb_t[ms][lane] = ct;
                ws.kb_i[ms][lane] = ci;
                ws.kb_a[ms][lane] = ca;
                ct = ot; ci = oi; ca = oa;
                mt = -INFINITY;
#pragma unroll 1
                for (int k = 0; k < K; ++k) {
                    const float t = ws.kb_t[k][lane];
                    if (t > mt) { mt = t; ms = k; }
                }
            }
        }
    }

    // ---- order the hits by ascending entry distance (kbuffer.cuh) ---------------------------------
    int maxcnt = cnt;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxcnt = max(maxcnt, __shfl_xor_sync(FULL, maxcnt, o));
    unsigned long long n_exact = 0;
    const unsigned long long perm = order_hits16(P, ws.kb_t, ws.kb_i, cnt, maxcnt, lane, pi, pj, n_exact);
    ST(S.st_f64 += n_exact);

    // ---- compositing: accum += T * alpha * rgb ; T *= 1 - alpha   (ray_tracer.py:96-98) ---------
    float T = 1.0f, cr = 0.0f, cg = 0.0f, cb = 0.0f, D = 0.0f;
    int nl = 0;
    if (maxcnt > 0) {
        float Y[15];
        float dx, dy, dz;
        sh_direction(cam, i0, j0, pi, pj, active, dx, dy, dz);
        sh_basis(dx, dy, dz, Y);
        const int nmine = min(cnt, P.depth);
        const int nloop = min(maxcnt, P.depth);
#pragma unroll 1
        for (int k = 0; k < nloop; ++k) {
            if (k < nmine && T >= P.t_cut) {
                const int slot = (int)((perm >> (4 * k)) & 15u);
                const int s = ws.kb_i[slot][lane];
                const float alpha = ws.kb_a[slot][lane];
                float r, g, b;
                eval_colour(P, s, Y, r, g, b);
                const float wgt = T * alpha;
                cr = fmaf(wgt, r, cr);
                cg = fmaf(wgt, g, cg);
                cb = fmaf(wgt, b, cb);
                T *= 1.0f - alpha;
                ++nl;
            }
        }
        if constexpr (DEPTH) {
            D = composite_depth(P, i0, j0, pi, pj, active, nmine, min(maxcnt, P.depth), [&](int k, int& s, float& a) {
                const int slot = (int)((perm >> (4 * k)) & 15u);
                s = ws.kb_i[slot][lane];
                a = ws.kb_a[slot][lane];
            });
        }
    }
    grant_wait(P, G);
    store_tile<DEPTH>(P, reinterpret_cast<float*>(&ws.rec[0][0]), lane, i0, j0, pi, pj, active, cr, cg, cb, T, D);
    tile_done(P, BC, tile, lane);
    if (active) {
        ST(S.st_rays += 1);
        ST(S.st_hit += nl > 0);
        ST(S.st_layers += (unsigned)nl);
    }
    ST(if (lane == 0) S.st_tiles += 1);

#undef ST
}

}  // namespace rtgs_dev
