// fused.cuh — k_render: the whole per-ray render path fused per tile (sm_100a).
//
//   camera ray generation        camera.py:31-71              (registers; rays never stored)
//   BVH traversal                scene.py:406-450             (warp-coherent frustum traversal)
//   ray-Gaussian intersection    gaussian.py:203-230          (local-frame quadratic)
//   response + SH colour         gaussian.py:140-201
//   front-to-back compositing    ray_tracer.py:79-104         (k-buffer of the `depth` nearest entries)
//
// Execution model.  A warp owns one 4x8-pixel tile at a time (lane = pixel) and pulls tiles from
// a global atomic counter (persistent threads).  All 32 primary rays share the camera origin, so
// the tile is a thin pyramid bounded by 4 planes through the origin.  The warp traverses the LBVH
// ONCE for the tile: up to 32 nodes are popped from a shared-memory stack per step, each lane
// tests the two child boxes of its node against the 4 planes, and survivors are compacted back with
// ballot/popc (internal children -> stack, the nearer one on top; leaves -> candidate queue).  Once rays hold
// K hits the traversal prunes by distance as well - the K-nearest form of the reference's far pruning
// (scene.py:417-419): a box beyond the farthest kept hit of every full ray that also misses the pyramid of the
// rays still lacking hits is dropped.  That makes this kernel the right one for tiles whose frustum holds
// thousands of Gaussians (lists_group sends it the groups whose list overflows).  Candidates are staged 32 at
// a time (one lane each, float64: origin shifted to the closest point of the tile's centre ray)
// and then every lane tests its own ray against every staged candidate with broadcast
// shared-memory reads: first a conservative 5-FMA quadratic (q - 3 as a polynomial of the pixel
// offset), then - in warp-wide rounds, one pending candidate per lane - the precise test, the entry
// distance and alpha.  Hits are appended to a per-lane K-entry buffer in shared memory (replace-max
// when full); after the traversal each lane ranks its entries and composites front to back.
//
// It renders depth > 16 (K = 32), RTGS_OPT_RENDER_MODE = 1, and - launched behind the list kernels - the tiles on
// the two hand-over lists.
//
// Numerics.  The reference's f32 formulation (B^2 - 4AC with a cofactor inverse) is ill-conditioned
// (SURVEY.md §7 hard part 1), and parity is defined against a float64 evaluation of the
// reference's maths.  The fast path is float32 but expressed relative to (Gaussian centre, tile
// centre ray), which keeps all magnitudes O(tile size / sigma); a hit/miss decision within a
// small band of the sqrt(3)-sigma surface, an entry distance within a band of 0, and adjacent
// k-buffer entries closer than a few ulp are re-evaluated in float64 from the raw parameters.
#pragma once
#include "kbuffer.cuh"

namespace rtgs_dev {
namespace fused {

constexpr int STACK_CAP = 512;
// Above STACK_SINGLE the traversal pops one node at a time (depth first).  A batch step grows the stack by <= 32 (two
// children per popped node), a single pop by <= 1 per level descended, i.e. by <= RTGS_MAX_TREE_DEPTH in all.
constexpr int STACK_SINGLE = STACK_CAP - 32 - RTGS_MAX_TREE_DEPTH;
constexpr int CQ_CAP = 96;
static_assert(STACK_SINGLE >= 64, "k_render: stack too small for batched traversal");
constexpr int BATCH = REC_BATCH;

struct __align__(16) TraversalScratch {
    StagedRecords rec;          // precise records (render_common.cuh: stage_candidate)
    float4 polyA[BATCH];        // coarse quadratics {c0 c1 c2 c3}
    float4 polyB[BATCH];        //                   {c4 c5 t_lo -}: t_lo = no ray of the tile enters the candidate before it
    int stack[STACK_CAP];
    int cq[CQ_CAP];
    Frustum open;               // pyramid of the rays that still lack hits (distance pruning, below)
};

template <int K>
struct __align__(16) WarpShared {
    union {
        TraversalScratch t;        // traversal phase
        struct {                   // compositing phase: hits in ascending entry distance
            int so_i[K][32];
            float so_a[K][32];
        } c;
    };
    float kb_t[K][32];     // per-lane hit buffer (unsorted): entry distance, sorted position, alpha
    int kb_i[K][32];
    float kb_a[K][32];
    int band_state[4];     // lane 0's band-completion counts (render_common.cuh: BandCount)
};

// STATS = true compiles the per-render counters in (rtgs_render with a stats pointer); the timed path
// uses STATS = false so that the 64-bit counters do not occupy registers.  DEPTH = true also composites the ray
// distance of every layer into P.out_depth (rtgs_render_depth; render_common.cuh: composite_depth).
template <int K, bool STATS, bool DEPTH = false>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, (K <= 16 ? 2 : 1)) k_render(const __grid_constant__ RenderParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpShared<K>& ws = reinterpret_cast<WarpShared<K>*>(smem_raw)[threadIdx.x >> 5];
    TraversalScratch& tr = ws.t;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const CamD& cam = P.cam;
    const int xe = P.x0 + P.w, ye = P.y0 + P.h;
    // work items: every tile id (cursor CTR_WORK2, as for the shading), or (fallback mode) the tiles the traversal,
    // then the shading handed over (cursor CTR_WORK3)
    const int n1 = P.use_fallback_list ? (int)min(P.counters[CTR_FALLBACK], (unsigned)P.ntiles) : 0;
    const int n2 = P.use_fallback_list ? (int)min(P.counters[CTR_FALLBACK2], (unsigned)P.ntiles) : 0;
    unsigned int* const cursor = P.counters + (P.use_fallback_list ? CTR_WORK3 : CTR_WORK2);

    if (P.use_fallback_list && blockIdx.x == 0 && threadIdx.x == 0) {
        // pool demand of this frame (for the host's sizing) and whether any frame so far needed the fallback
        *reinterpret_cast<volatile int*>(P.mirror) = (int)min(P.counters[CTR_POOL], 0x7fffffffu);
        if (P.counters[CTR_FALLBACK] != 0) *reinterpret_cast<volatile int*>(P.mirror + 1) = 1;
    }

    PeerGrant grant;
    BandCount band_count;
    grant_begin(P, grant);
    band_begin(P, band_count, ws.band_state, lane);
    unsigned long long st_nodes = 0, st_cands = 0, st_pairs = 0, st_f64 = 0, st_layers = 0, st_hit = 0,
                       st_rays = 0, st_tiles = 0, st_steps = 0, st_ins = 0;
    unsigned st_max_stack = 0;
#define ST(expr) do { if (STATS) { expr; } } while (0)

#pragma unroll 1
    for (;;) {
        int tile = 0;
        if (lane == 0) {
            tile = (int)atomicAdd(cursor, 1u);
            if (P.use_fallback_list) tile = tile < n1 ? P.fallback_tiles[tile] : (tile - n1 < n2 ? P.fallback_tiles2[tile - n1] : P.ntiles);
            else tile = work_to_id(P, tile, P.macro_cols * TILES_PER_MACRO, P.ntiles);
        }
        tile = __shfl_sync(FULL, tile, 0);
        if (tile >= P.ntiles) break;
        band_claim(P, band_count, tile, lane);
        int i0, j0;
        if (!tile_origin(P, tile, i0, j0) || i0 >= xe || j0 >= ye) {
            tile_done(P, band_count, tile, lane);
            continue;
        }
        const int pi = i0 + lane / TILE_J, pj = j0 + lane % TILE_J;
        const bool active = pi < xe && pj < ye;

        TileRays ry;
        make_tile_rays(cam, i0, j0, pi, pj, active, ry);
        // Distance pruning compares Euclidean box distances with ray parameters: distance = t |d|, and |d| is 1 only
        // for a unit camera quaternion (the reference uses the rotation as given, camera.py:52).  len_max = the longest
        // direction among the tile's rays (corners and centre, with a margin for the rays in between).
        float len_max;
        {
            const d3 dc = cam_dir(cam, (double)i0 + 0.5 * TILE_I, (double)j0 + 0.5 * TILE_J);   // tile-centre ray
            double l2 = d3dot(dc, dc);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const d3 e = cam_dir(cam, (double)(i0 + (k & 1) * TILE_I), (double)(j0 + (k >> 1) * TILE_J));
                l2 = fmax(l2, d3dot(e, e));
            }
            len_max = (float)(sqrt(l2) * 1.0001);
        }
        Frustum fr;
        make_frustum(cam, i0, i0 + TILE_I, j0, j0 + TILE_J, fr);

        // ---- per-lane hit buffer (shared memory, unsorted; replace-max once K entries are held) --
        int cnt = 0;
        float kmax_t = INFINITY;
        int kmax_slot = 0;

        // Transmittance exhaustion (t_cut > 0, K = 16): once the hits a ray holds bring its transmittance below
        // t_cut, nothing behind the hit that does so is ever composited (ray_tracer.py:96-98 with the early-out), and
        // hits found later can only lower the transmittance further.  d_T is that hit's entry distance (with a margin);
        // the ray is then CLOSED at min(d_T, farthest of K kept hits) exactly like a ray whose buffer is full.
        float d_T = INFINITY;
        bool kb_dirty = false;         // the lane's buffer changed since d_T was last evaluated

        // Distance pruning - the K-nearest form of the reference's "skip a node whose entry distance exceeds the best
        // hit so far" (scene.py:417-419).  A ray that holds K hits needs nothing farther than its farthest one, so a
        // box is dropped when it lies beyond `cut` = the largest such distance among the rays that are full (with a
        // margin far above float32 rounding, so that near-ties at the K-th place still see both contenders) AND
        // misses the pyramid of the rays that are not full yet (`tr.open`, the bounding pixel rectangle of those
        // rays; initially the whole tile).  Children are pushed far one first.  This is what keeps a tile that looks
        // along a surface - thousands of splats in its frustum, the first few dozen of them opaque - affordable.
        float cut2 = -1.0f;            // (cut * (1 + 1e-4))^2, < 0: no ray is full yet
        unsigned open_mask = __ballot_sync(FULL, active);
        bool open_all = true;          // tr.open == fr
        const float ox = (float)cam.o[0], oy = (float)cam.o[1], oz = (float)cam.o[2];
        auto box_dist2 = [&](float cx, float cy, float cz, float hx, float hy, float hz) {
            const float dx = fmaxf(fabsf(ox - cx) - hx, 0.0f), dy = fmaxf(fabsf(oy - cy) - hy, 0.0f),
                        dz = fmaxf(fabsf(oz - cz) - hz, 0.0f);
            return dx * dx + dy * dy + dz * dz;
        };

        int top = 1, ncq = 0;
        if (lane == 0) tr.stack[0] = 0;
        __syncwarp();

        // ================================ traversal ==========================================
#pragma unroll 1
        while (top > 0 || ncq > 0) {
            if (top > 0) {
                const int take = top > STACK_SINGLE ? 1 : min(32, top);
                int node = -1;
                if (lane < take) node = tr.stack[top - 1 - lane];
                top -= take;
                __syncwarp();
                bool h0 = false, h1 = false;
                int c0 = 0, c1 = 0;
                if (node >= 0) {
                    float4 a, b, c, d;
                    ldg256(P.nodes + (int64_t)node * 4 + 0, a, b);
                    ldg256(P.nodes + (int64_t)node * 4 + 2, c, d);
                    c0 = __float_as_int(d.x);
                    c1 = __float_as_int(d.y);
                    h0 = box_in_frustum(fr, a.x, a.y, a.z, a.w, b.x, b.y);
                    h1 = box_in_frustum(fr, b.z, b.w, c.x, c.y, c.z, c.w);
                    const float d0 = box_dist2(a.x, a.y, a.z, a.w, b.x, b.y);
                    const float d1 = box_dist2(b.z, b.w, c.x, c.y, c.z, c.w);
                    if (cut2 >= 0.0f) {
                        if (h0 && d0 > cut2)
                            h0 = open_mask != 0 && (open_all || box_in_frustum(tr.open, a.x, a.y, a.z, a.w, b.x, b.y));
                        if (h1 && d1 > cut2)
                            h1 = open_mask != 0 && (open_all || box_in_frustum(tr.open, b.z, b.w, c.x, c.y, c.z, c.w));
                    }
                    if (d1 > d0) {   // child 1 is pushed last, i.e. popped first: make it the nearer one
                        const int ci = c0; c0 = c1; c1 = ci;
                        const bool hi = h0; h0 = h1; h1 = hi;
                    }
                }
                ST(st_nodes += 2ull * (unsigned)take);
                ST(st_steps += 1);
                const unsigned mI0 = __ballot_sync(FULL, h0 && c0 >= 0), mI1 = __ballot_sync(FULL, h1 && c1 >= 0);
                const unsigned mL0 = __ballot_sync(FULL, h0 && c0 < 0), mL1 = __ballot_sync(FULL, h1 && c1 < 0);
                if (h0 && c0 >= 0) tr.stack[top + __popc(mI0 & lt_mask)] = c0;
                const int topa = top + __popc(mI0);
                if (h1 && c1 >= 0) tr.stack[topa + __popc(mI1 & lt_mask)] = c1;
                top = topa + __popc(mI1);
                if (h0 && c0 < 0) tr.cq[ncq + __popc(mL0 & lt_mask)] = ~c0;
                const int ncqa = ncq + __popc(mL0);
                if (h1 && c1 < 0) tr.cq[ncqa + __popc(mL1 & lt_mask)] = ~c1;
                ncq = ncqa + __popc(mL1);
                ST(st_max_stack = max(st_max_stack, (unsigned)top));
                __syncwarp();
            }
            // -------- candidate batch: stage (one lane each, float64) then test (all lanes) --
#pragma unroll 1
            while (ncq >= BATCH || (top == 0 && ncq > 0)) {
                const int m = min(BATCH, ncq);
                ncq -= m;
                const int m4 = (m + 3) & ~3;
                if (lane < m) {
                    float4 rec[REC_QUADS];
                    float poly[6], t_lo;
                    stage_candidate<true>(P, ry, tr.cq[ncq + lane], rec, poly, t_lo);
#pragma unroll
                    for (int k = 0; k < REC_QUADS; ++k) tr.rec[k][lane] = rec[k];
                    tr.polyA[lane] = make_float4(poly[0], poly[1], poly[2], poly[3]);
                    tr.polyB[lane] = make_float4(poly[4], poly[5], t_lo, 0.0f);
                } else if (lane < m4) {   // pad to a multiple of 4: never a candidate
                    tr.polyA[lane] = make_float4(1.0f, 0.0f, 0.0f, 0.0f);
                    tr.polyB[lane] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                }
                __syncwarp();
                ST(st_cands += (unsigned)m);
                ST(st_pairs += 32ull * (unsigned)m);
                // ---- coarse: mask of the staged candidates this ray may hit (as in shade.cuh) ----------
                // a closed ray takes nothing that certainly begins behind its cut (margin: near ties at the K-th
                // place are decided in float64 by the insertion code, so they must reach it)
                const float my_cut = fminf(cnt == K ? kmax_t : INFINITY, d_T) * 1.000004f;
                unsigned mask = 0;
#pragma unroll 1
                for (int c = 0; c < m4; c += 4) {
                    unsigned nib = 0;
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float4 pA = tr.polyA[c + u];
                        const float4 pB = tr.polyB[c + u];
                        const float ta = fmaf(ry.pa, pA.w, fmaf(ry.pb, pB.x, pA.y));   // c1 + a c3 + b c4
                        const float tb = fmaf(ry.pb, pB.y, pA.z);                      // c2 + b c5
                        const float S = fmaf(ry.pa, ta, fmaf(ry.pb, tb, pA.x));
                        if (S < 0.0f && pB.z <= my_cut) nib |= 1u << u;
                    }
                    mask |= nib << c;
                }
                if (!active) mask = 0;
                // ---- precise: warp-wide rounds, one candidate per lane and round ----------------------
#pragma unroll 1
                while (__any_sync(FULL, mask != 0)) {
                    if (mask != 0) {
                        const int c = __ffs(mask) - 1;
                        mask &= mask - 1;
                        const PreciseHit h = precise_test(P, tr.rec, c, ry, pi, pj);
                        ST(st_f64 += h.refined);
                        if (h.hit && h.t1 <= d_T) {
                            kb_dirty = true;
                            auto find_farthest = [&]() {
                                float mt = -INFINITY;
                                int ms = 0;
#pragma unroll 4
                                for (int k = 0; k < K; ++k) {
                                    const float t = ws.kb_t[k][lane];
                                    if (t > mt) { mt = t; ms = k; }
                                }
                                kmax_t = mt;
                                kmax_slot = ms;
                            };
                            if (cnt < K) {
                                const int slot = cnt++;
                                ws.kb_t[slot][lane] = h.t1;
                                ws.kb_i[slot][lane] = h.s;
                                ws.kb_a[slot][lane] = h.alpha;
                                if (cnt == K) find_farthest();
                            } else {
                                // full: the candidate replaces the farthest entry if it is nearer.  Whenever
                                // two contenders for the last place are within float32 rounding of each other
                                // - the candidate and the farthest entry, or the evicted entry and the new
                                // farthest one - their float64 entry distances decide (exact_less; rare).
                                float ct = h.t1, ca = h.alpha;
                                int cs = h.s;
#pragma unroll 1
                                for (;;) {
                                    bool nearer = ct < kmax_t;
                                    if (fabsf(ct - kmax_t) <= 2e-6f * kmax_t) {
                                        nearer = exact_less(P.raw, cam, cs, ws.kb_i[kmax_slot][lane], pi, pj);
                                        ST(st_f64 += 2);
                                    }
                                    if (!nearer) break;
                                    const float et = kmax_t, ea = ws.kb_a[kmax_slot][lane];
                                    const int es = ws.kb_i[kmax_slot][lane];
                                    ws.kb_t[kmax_slot][lane] = ct;
                                    ws.kb_i[kmax_slot][lane] = cs;
                                    ws.kb_a[kmax_slot][lane] = ca;
                                    find_farthest();
                                    if (!(et - kmax_t <= 2e-6f * et)) break;
                                    ct = et; cs = es; ca = ea;   // the evicted entry ties with the new farthest
                                }
                            }
                        }
                    }
                    ST(st_ins += 1);
                }
                __syncwarp();
                // ---- pruning state after the batch: which rays are closed, and how far they still look ----
                {
                    if constexpr (K == 16) {
                        if (P.t_cut > 0.0f && __any_sync(FULL, kb_dirty)) {
                            // order the lane's hits (truncated keys are enough: the margin below covers near ties)
                            // and multiply the transmittance through
                            unsigned key[16];
#pragma unroll
                            for (int k = 0; k < 16; ++k)
                                key[k] = k < cnt ? ((__float_as_uint(ws.kb_t[k][lane]) & ~15u) | (unsigned)k) : 0xffffffffu;
                            sort_keys<16>(key);
                            const float lim = 0.99f * P.t_cut;
                            float Tacc = 1.0f, d = INFINITY;
#pragma unroll
                            for (int r = 0; r < 16; ++r) {
                                if (r < cnt && d == INFINITY) {
                                    const int slot = (int)(key[r] & 15u);
                                    Tacc *= 1.0f - ws.kb_a[slot][lane];
                                    if (Tacc < lim) d = ws.kb_t[slot][lane];
                                }
                            }
                            d_T = d * 1.0001f;     // (inf stays inf)
                            kb_dirty = false;
                        }
                    }
                    const float c_ray = fminf(cnt == K ? kmax_t : INFINITY, d_T);
                    const bool closed = active && c_ray < INFINITY;
                    float cm = closed ? c_ray : -1.0f;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) cm = fmaxf(cm, __shfl_xor_sync(FULL, cm, o));
                    if (cm >= 0.0f) {
                        cm *= 1.0001f * len_max;     // ray parameter -> distance
                        cut2 = cm * cm;
                    }
                    const bool open = active && !closed;
                    const unsigned om = __ballot_sync(FULL, open);
                    if (om != open_mask) {
                        open_mask = om;
                        if (om != 0) {
                            int il = open ? pi : 0x7fffffff, ih = open ? pi : -1;
                            int jl = open ? pj : 0x7fffffff, jh = open ? pj : -1;
#pragma unroll
                            for (int o = 16; o > 0; o >>= 1) {
                                il = min(il, __shfl_xor_sync(FULL, il, o));
                                ih = max(ih, __shfl_xor_sync(FULL, ih, o));
                                jl = min(jl, __shfl_xor_sync(FULL, jl, o));
                                jh = max(jh, __shfl_xor_sync(FULL, jh, o));
                            }
                            Frustum fo;
                            make_frustum(cam, il, ih + 1, jl, jh + 1, fo);
                            if (lane == 0) tr.open = fo;
                            open_all = false;
                        }
                        __syncwarp();
                    }
                }
            }
        }

        int maxcnt = cnt;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) maxcnt = max(maxcnt, __shfl_xor_sync(FULL, maxcnt, o));
        __syncwarp();
        float T = 1.0f, cr = 0.0f, cg = 0.0f, cb = 0.0f, D = 0.0f;
        int nl = 0;
        if constexpr (K == 16) {
            // ---- order the hits (bitonic network over register keys, near ties by float64: kbuffer.cuh) and composite
            // accum += T * alpha * rgb ; T *= 1 - alpha   (ray_tracer.py:96-98), rgb = color + eval_sh(normalize(dir))
            unsigned long long n_exact = 0;
            const unsigned long long perm = order_hits16(P, ws.kb_t, ws.kb_i, cnt, maxcnt, lane, pi, pj, n_exact);
            ST(st_f64 += n_exact);
            float Y[15];
            {
                float dx, dy, dz;
                sh_direction(cam, i0, j0, pi, pj, active, dx, dy, dz);
                sh_basis(dx, dy, dz, Y);
            }
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
                D = composite_depth(P, i0, j0, pi, pj, active, nmine, nloop, [&](int k, int& s, float& a) {
                    const int slot = (int)((perm >> (4 * k)) & 15u);
                    s = ws.kb_i[slot][lane];
                    a = ws.kb_a[slot][lane];
                });
            }
            __syncwarp();
        } else {
            // ---- K = 32: rank counting into the compositing list.  rank_i = #{j : t_j < t_i}; pairs within float32
            // rounding of each other are ordered by their float64 entry distances (exact_less).
            if (maxcnt > 0) {
                float tk[K];
#pragma unroll
                for (int k = 0; k < K; ++k) tk[k] = k < cnt ? ws.kb_t[k][lane] : INFINITY;
#pragma unroll 1
                for (int i = 0; i < maxcnt; ++i) {
                    if (i < cnt) {
                        const float ti_ = ws.kb_t[i][lane];
                        const float band = 2e-6f * fabsf(ti_);
                        int rank = 0, nnear = 0;
#pragma unroll
                        for (int j = 0; j < K; ++j) {
                            rank += tk[j] < ti_;
                            nnear += fabsf(tk[j] - ti_) <= band;
                        }
                        const int id = ws.kb_i[i][lane];
                        if (nnear > 1) {   // rare: resolve near ties exactly
                            rank = 0;
#pragma unroll 1
                            for (int j = 0; j < cnt; ++j) {
                                if (j == i) continue;
                                const float tj_ = ws.kb_t[j][lane];
                                if (fabsf(tj_ - ti_) <= band) {
                                    rank += exact_less(P.raw, cam, ws.kb_i[j][lane], id, pi, pj);
                                    ST(st_f64 += 2);
                                } else {
                                    rank += tj_ < ti_;
                                }
                            }
                        }
                        ws.c.so_i[rank][lane] = id;
                        ws.c.so_a[rank][lane] = ws.kb_a[i][lane];
                    }
                }
            }
            __syncwarp();
            // ================================ compositing ========================================
            // accum += T * alpha * rgb ; T *= 1 - alpha   (ray_tracer.py:96-98), rgb = color +
            // eval_sh(normalize(dir)) (gaussian.py:199-200).
            {
                float Y[15];
                {
                    float dx, dy, dz;
                    sh_direction(cam, i0, j0, pi, pj, active, dx, dy, dz);
                    sh_basis(dx, dy, dz, Y);
                }
                const int nmine = min(cnt, P.depth);
                const int nloop = min(maxcnt, P.depth);
#pragma unroll 1
                for (int k = 0; k < nloop; ++k) {
                    if (k < nmine && T >= P.t_cut) {
                        const int s = ws.c.so_i[k][lane];
                        const float alpha = ws.c.so_a[k][lane];
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
                    D = composite_depth(P, i0, j0, pi, pj, active, nmine, nloop, [&](int k, int& s, float& a) {
                        s = ws.c.so_i[k][lane];
                        a = ws.c.so_a[k][lane];
                    });
                }
            }
        }
        grant_wait(P, grant);
        store_tile<DEPTH>(P, reinterpret_cast<float*>(&ws.kb_t[0][0]), lane, i0, j0, pi, pj, active, cr, cg, cb, T, D);
        tile_done(P, band_count, tile, lane);
        if (active) {
            ST(st_rays += 1);
            ST(st_hit += nl > 0);
            ST(st_layers += (unsigned)nl);
        }
        ST(if (lane == 0) st_tiles += 1);
    }

    band_flush(P, band_count, lane);
    if (STATS && P.stats) {
        unsigned long long v[ST_COUNT] = {0};
        v[ST_RAYS] = st_rays; v[ST_RAYS_HIT] = st_hit; v[ST_LAYERS] = st_layers; v[ST_F64] = st_f64;
        // warp-uniform counters are taken from lane 0 only
        if (lane == 0) {
            v[ST_NODES] = st_nodes;
            v[ST_CANDS] = st_cands;
            v[ST_PAIRS] = st_pairs;
            v[ST_TILES] = st_tiles;
            v[ST_STEPS] = st_steps;
            v[ST_INSERTS] = st_ins;
            v[ST_FALLBACK] = P.use_fallback_list ? st_tiles : 0;
        }
#pragma unroll
        for (int k = 0; k < ST_COUNT; ++k) {
            unsigned long long x = v[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
            if (lane == 0 && x) atomicAdd(P.stats + k, x);
        }
        if (lane == 0) atomicMax(P.stats + ST_MAX_FUSED_STACK, (unsigned long long)st_max_stack);
    }
    if (P.final_kernel) cta_finish(P, CTR_DONE2);
}
#undef ST


}  // namespace fused
}  // namespace rtgs_dev
