// common.cuh — shared declarations for the B200-native rtgs render path (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/rtgs_b200.h"

#define RTGS_SM_COUNT_FALLBACK 148
#define RTGS_MAX_BANDS 32
// Deepest leaf the traversal stacks are sized for: 62 levels for unique (30-bit code, index) keys, 63 + 30 for
// 63-bit codes with repeats (lbvh.cu: k_karras<DUP>, k_max_depth); the build refuses anything deeper.
#define RTGS_MAX_TREE_DEPTH 96

// ---- error plumbing (never abort across the ABI) ---------------------------------------------
void rtgs_set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            rtgs_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,   \
                           __LINE__);                                                          \
            return RTGS_ERR_CUDA;                                                              \
        }                                                                                      \
    } while (0)

#define RTGS_CHECK_ARG(cond)                                                                   \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            rtgs_set_error("invalid argument: %s (%s:%d)", #cond, __FILE__, __LINE__);         \
            return RTGS_ERR_INVALID;                                                           \
        }                                                                                      \
    } while (0)

// ---- device data layout (all records 16-byte aligned SoA of float4) ---------------------------
// Everything below is stored in MORTON-SORTED order (sorted position s), so that neighbouring
// BVH leaves are neighbours in memory.
//
// geo  [s*4 + 0] = { p.x, p.y, p.z, opacity }
//      [s*4 + 1] = { W00, W01, W02, W10 }        W = S^-1 R^T / |q|^4  (local-frame matrix:
//      [s*4 + 2] = { W11, W12, W20, W21 }        x' = W (x - p);  Sigma^-1 = W^T W)
//      [s*4 + 3] = { W22, dc.r, dc.g, dc.b }     dc = post-sigmoid colour (scene.py:113)
// shp  [s*12 .. s*12+11] = 45 SH floats (sh_10.rgb, sh_11.rgb, ... sh_36.rgb) + dc.rgb
// raw  [s*3 .. s*3+2]    = { p.xyz, q.x } { q.yzw, s.x } { s.yz, original index (int bits), 0 }
//                          (inputs of the float64 exact-decision path)
// node [k*4 + 0] = { lc.x, lc.y, lc.z, lh.x }      child boxes as (centre c, half extent h), h rounded up
//      [k*4 + 1] = { lh.y, lh.z, rc.x, rc.y }
//      [k*4 + 2] = { rc.z, rh.x, rh.y, rh.z }
//      [k*4 + 3] = { left, right (int bits), 0, 0 }   child >= 0: internal node id;
//                                                      child <  0: leaf, sorted position = ~child
// leafbox [s*2] = { p.xyz, h.x } { h.yz, fp16 rho_xy rho_xz, fp16 rho_yz 0 }   leaf records by sorted position:
//                 exact centre, half extents of the sqrt(3)-sigma ellipsoid, correlations of Sigma
struct rtgs_scene {
    int device = 0;
    int64_t n = 0;
    bool has_sh = false;
    bool built = false;
    int sm_count = RTGS_SM_COUNT_FALLBACK;

    // stored parameters, ORIGINAL order (Scene.gaussian_field)
    float* pos = nullptr;      // n*3
    float* rot = nullptr;      // n*4
    float* scale = nullptr;    // n*3
    float* color = nullptr;    // n*3
    float* opacity = nullptr;  // n
    float* sh = nullptr;       // n*45 or null

    // LBVH integers (parity read-back) and boxes
    uint32_t* morton = nullptr;      // n, original order
    uint64_t* morton64 = nullptr;    // n, original order: 63-bit codes (RTGS_OPT_MORTON_BITS = 63 only)
    int opt_morton_bits = 0;         // RTGS_OPT_MORTON_BITS: 0 = automatic, 30, 63
    int morton_bits_used = 30;       // width of the codes the current tree was built from
    int64_t distinct_codes = -1;     // distinct 30-bit codes found by the last 30-bit build
    uint32_t* sorted_idx = nullptr;  // n
    int32_t* child = nullptr;        // (n-1)*2 unified ids
    int32_t* parent = nullptr;       // 2n-1
    float* aabb = nullptr;           // (2n-1)*6
    float bounds[6] = {0, 0, 0, 0, 0, 0};

    // packed render records
    float4* geo = nullptr;
    float4* shp = nullptr;
    cudaTextureObject_t geo_tex = 0;   // (experiment) geo as a linear float4 texture
    cudaTextureObject_t shp_tex = 0;   // shp as a linear float4 texture (eval_colour); 0 when the scene exceeds one texture
    float4* raw = nullptr;
    float4* nodes = nullptr;
    float4* leafbox = nullptr;   // n*2: leaf box (centre, half extent) by sorted position
    float4* nodes4 = nullptr;    // num_nodes*8: two-level nodes (records of both children), k_tile_lists
    int64_t num_nodes = 0;  // max(n-1, 1)
    float build_ms = 0.0f;  // device time of the last LBVH build (Morton codes ... packed nodes)
    int max_depth = 0;      // depth of the deepest leaf of the current tree (root = 0)

    // render scratch.  A frame's work counters and candidate lists live in a FrameScratch; a scene has two, so
    // that frames launched on two alternating streams overlap on the device (frame f+1's traversal fills the SMs
    // that frame f's shading tail leaves idle) instead of being serialised by the library.
    struct FrameScratch {
        unsigned int* counters = nullptr;     // CTR_COUNT: work counters, pool cursor, fallback count
        void* tile_desc = nullptr;            // candidate lists (render_common.cuh), sized on first use
        int* list_pool = nullptr;
        int* fallback_tiles = nullptr;
        int* fallback_tiles2 = nullptr;
        unsigned int* ready = nullptr;        // per traversal group: sequence number of the frame whose lists are complete
        unsigned int frame_seq = 0;           // frames launched through k_frame so far (ready[] is compared with it)
        bool counters_dirty = false;          // the last frame did not zero the work counters itself
        int list_tiles = 0;
        int pool_chunks = 0;
        int* mirror = nullptr;                // mapped pinned host memory: [0] pool demand of the last finished frame,
        int* mirror_dev = nullptr;            //                            [1] some finished frame had fallback tiles,
                                              //                            [2] some frame had heavy groups (k_heavy_lists)
        int* heavy_groups = nullptr;          // depth-capped lists (heavy_lists.cuh): queue of heavy groups, per-tile caps,
        float* tile_cap = nullptr;            // per-warp lists of deferred nodes; sized with the candidate lists / on first use
        int2* heavy_scratch = nullptr;
        int heavy_scratch_warps = 0;
        cudaEvent_t free_event = nullptr;     // behind the last frame that used this scratch
        cudaStream_t stream = nullptr;        // the stream that frame was launched on
        bool used = false;
        uint64_t last_use = 0;
    };
    FrameScratch scratch[2];
    uint64_t scratch_clock = 0;
    bool exclusive_inflight = false;         // the last frame launched used the once-only counters (statistics, bands)
    unsigned long long* stats_dev = nullptr;  // 12 counters
    // multi-GPU hand-over of the NEXT frame (rtgs_scene_set_frame_sync; cleared when that frame is launched)
    unsigned int* sync_arrive = nullptr;
    const unsigned int* sync_grant = nullptr;
    unsigned int sync_grant_value = 0;
    int64_t opt_pool_chunks = -1;             // RTGS_OPT_LIST_POOL_CHUNKS (-1 = default sizing)
    int opt_stripe_mod = 1, opt_stripe_rem = 0;   // RTGS_OPT_STRIPE
    int opt_render_mode = -1;                 // RTGS_OPT_RENDER_MODE (-1 = RTGS_RENDER_MODE env or 0)
    int opt_heavy_lists = -1;                 // RTGS_OPT_HEAVY_LISTS (-1 = RTGS_HEAVY_SLAB env or 1)
    int opt_heavy_limit = -1;                 // RTGS_OPT_HEAVY_LIMIT (-1 = RTGS_HEAVY_LIMIT env or the shared-memory capacity)
    // rtgs_render_host: device staging + band flags, double-buffered so that two frames can be in flight
    // (rtgs_render_host_submit / _collect: frame f+1 renders while the last bands of frame f are copied out)
    struct HostSlot {
        float* stage_rgb = nullptr;
        float* stage_T = nullptr;
        size_t stage_pixels = 0;
        void* stage_packed = nullptr;         // compact delivery (RTGS_PIXELS_F16 / _RGBA8): the converted image
        size_t stage_packed_pixels = 0;
        int* flags = nullptr;                 // this slot's part of band_flags (host / device alias)
        int* flags_dev = nullptr;
        cudaEvent_t done = nullptr;           // recorded behind the frame's last kernel
        cudaEvent_t copied = nullptr;         // recorded behind the frame's whole-image DMA (pipelined delivery)
        int nb = 0, bmc = 0, sched = 0, w = 0, h = 0;
        float* host_rgb = nullptr;
        float* host_T = nullptr;
    };
    HostSlot host_slot[2];
    int host_head = 0, host_inflight = 0;     // next slot to submit into; frames submitted and not collected
    int* band_flags_cur_dev = nullptr;        // flags of the frame being launched (set around rtgs_launch_render)
    float* pinned_rgb = nullptr;
    float* pinned_T = nullptr;
    size_t pinned_pixels = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t own_stream2 = nullptr;       // pipelined delivery: the two frames in flight render on alternating streams
    cudaStream_t copy_stream = nullptr;       // framebuffer DMA of rtgs_render_host, overlapping the render
    cudaStream_t copy_stream2 = nullptr;      // second DMA queue (bands alternate, hiding the per-copy set-up)
    unsigned int* band_done = nullptr;        // device: finished tile ids per band
    int* band_flags = nullptr;                // mapped pinned host memory: band complete
    int* band_flags_dev = nullptr;            // device alias of band_flags
    int bands_active = 0;                     // set by rtgs_render_host around its launch
    int band_macro_cols = 0;
    int band_schedule = 0;                    // macro-column order of the banded launch (render_common.cuh)

    // per-kernel timing ring (RTGS_OPT_KERNEL_TIMING): 4 events per frame slot
    std::vector<cudaEvent_t> timing_events;
    std::vector<unsigned char> timing_ran;   // per slot: bit k = kernel k was launched
    int64_t timing_frames = 0;               // renders recorded since timing was switched on
};

// ---- launchers implemented in the kernel translation units ------------------------------------
int rtgs_lbvh_build(rtgs_scene* s);   // lbvh.cu
int rtgs_launch_render(rtgs_scene* s, const rtgs_camera* cam, int x0, int y0, int w, int h,
                       int depth, float t_cut, int accumulate, int full_pitch, float* out_rgb,
                       float* out_T, cudaStream_t stream, bool want_stats);  // render.cu
int rtgs_heavy_lists_mode(const rtgs_scene* s);
int rtgs_launch_render_backward(rtgs_scene* s, const rtgs_camera* cam, int x0, int y0, int w, int h, int depth,
                                float t_cut, const float* dL_drgb, const float* dL_dT, float* const grads[6],
                                float* const cam_grads[3], float* replay_rgb, float* replay_T,
                                cudaStream_t stream);  // render.cu (backward.cuh)
int rtgs_launch_render_rays(rtgs_scene* s, int64_t nrays, const float* rays, int depth, float t_cut, float* out_rgb,
                            float* out_T, cudaStream_t stream);  // render.cu (backward.cuh)
int rtgs_launch_render_rays_backward(rtgs_scene* s, int64_t nrays, const float* rays, int depth, float t_cut,
                                     const float* dL_drgb, const float* dL_dT, float* const grads[6], float* grad_rays,
                                     float* replay_rgb, float* replay_T, cudaStream_t stream);
int rtgs_launch_generate_rays(const rtgs_camera* cam, float* rays, cudaStream_t stream);
int rtgs_launch_trace_closest(rtgs_scene* s, int64_t nrays, const float* rays, int32_t* idx,
                              float* t12, cudaStream_t stream);
int rtgs_launch_wait_counter(const unsigned int* counter, unsigned int value, cudaStream_t stream);
int rtgs_launch_set_counter(unsigned int* counter, unsigned int value, cudaStream_t stream);
int rtgs_launch_store_u32(unsigned int* counter, unsigned int value, cudaStream_t stream);
int rtgs_launch_add_counter(unsigned int* counter, cudaStream_t stream);
int rtgs_launch_pack_pixels(const float* rgb, void* out, int64_t npix, int format, cudaStream_t stream);
int rtgs_launch_activate_ply(int64_t n, const float* rows_dev, int stride, const int32_t* col,
                             float scale, int sh_layout, float* pos, float* rot, float* sca,
                             float* color, float* opacity, float* sh, cudaStream_t stream);
