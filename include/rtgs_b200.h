/*
 * rtgs_b200.h — C-ABI of the B200-native rtgs per-ray render path.
 *
 * The reference (fangjunzhou/rt-gaussian-splat-renderer, Python + Taichi) has no FFI layer: its
 * boundary is the Python object API  Scene / Camera / RayTracer.  This header is the C boundary a
 * binding for that API calls into (the Python mirror in rt-gaussian-splat-renderer_b200/rtgs/ does
 * so through ctypes; INTEGRATION.md shows the stub).  Each entry point cites the reference
 * interface (file:line under /root/reference) that it replaces.
 *
 * Conventions
 *  - every function returns RTGS_OK (0) or a negative rtgs_status; nothing throws or aborts across
 *    the ABI; rtgs_last_error() returns a thread-local message for the last failure.
 *  - plain pointers and sizes only.  "host" pointers are ordinary host memory borrowed for the
 *    duration of the call; "device" pointers are CUDA device memory on the scene's device.
 *  - a scene handle is bound to one CUDA device; calls on one handle must not overlap; different
 *    handles may be driven concurrently from different host threads.
 *  - image layout is the reference's field layout: pixel (i,j) = (column from the left, row from
 *    the BOTTOM), shape (W,H), i-major (index i*H + j)  (camera.py:33-35,67-70; ray_tracer.py:33-37).
 *  - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).
 */
#ifndef RTGS_B200_H
#define RTGS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTGS_ABI_VERSION 3
#define RTGS_MAX_DEPTH 32        /* largest `depth` rtgs_render composites in one pass */

typedef enum rtgs_status {
    RTGS_OK = 0,
    RTGS_ERR_INVALID = -1,       /* bad argument */
    RTGS_ERR_CUDA = -2,          /* a CUDA runtime call failed (message has the CUDA error) */
    RTGS_ERR_STATE = -3,         /* call order: e.g. render before build_bvh */
    RTGS_ERR_NOMEM = -4
} rtgs_status;

typedef struct rtgs_scene rtgs_scene;      /* opaque; owns all device memory */

/* Camera — camera.py:17-29 (position, rotation quaternion (x,y,z,w), buf_size, focal_length).
 * `rotation` is used as given (not re-normalised), as in Camera.generate_ray (camera.py:52). */
typedef struct rtgs_camera {
    float position[3];
    float rotation[4];
    float focal[2];
    int32_t width, height;
} rtgs_camera;

/* Per-render counters (optional; mean values are over the rays of the rendered region). */
typedef struct rtgs_render_stats {
    uint64_t rays;               /* pixels rendered */
    uint64_t rays_hit;           /* rays with >= 1 composited Gaussian */
    uint64_t layers;             /* total composited layers (sum over rays of min(hits, depth)) */
    uint64_t nodes_tested;       /* BVH child boxes tested against tile frusta */
    uint64_t candidates;         /* (tile, Gaussian) candidates staged */
    uint64_t pair_tests;         /* ray-Gaussian intersection tests */
    uint64_t f64_refinements;    /* borderline decisions re-evaluated in float64 */
    uint64_t tiles;              /* warp tiles processed */
    uint64_t traversal_steps;    /* warp-wide traversal iterations (each pops <= 32 nodes) */
    uint64_t insert_rounds;      /* warp-wide k-buffer insertion rounds */
    uint64_t fallback_tiles;     /* tiles rendered by the fused kernel because their list did not fit the pool */
    uint64_t useful_candidates;  /* staged candidates that passed the coarse test for at least one ray */
    /* high-water marks of the render (maxima over all warps): the traversal stacks are bounded by construction
     * (DESIGN.md §4: 256 entries in the list traversal, 512 in the fused kernel, for trees up to 96 levels deep);
     * these let a test assert the bounds on the device */
    uint64_t max_lists_stack;    /* deepest stack of the list traversal (entries) */
    uint64_t max_fused_stack;    /* deepest stack of the fused kernel (entries) */
    uint64_t max_group_list;     /* longest shared-memory candidate list of an 8x16-pixel group (<= 960) */
    /* depth-capped lists of heavy groups (RTGS_OPT_HEAVY_LISTS, csrc/heavy_lists.cuh) */
    uint64_t heavy_groups;       /* 4x8-pixel tiles listed in depth slabs (their group's frustum overflows the shared list) */
    uint64_t heavy_failed;       /* ... of them handed on to the fused kernel (slab or deferred list overflowed) */
    uint64_t heavy_passes;       /* cap raises, summed over the heavy groups */
    uint64_t heavy_sample_tests; /* candidates run through the hit test by k_heavy_lists */
    uint64_t max_deferred;       /* longest list of deferred nodes (<= 2048) */
    uint64_t heavy_retries;      /* passes repeated with a smaller step because the slab overflowed the shared list */
    uint64_t heavy_failed_list;      /* heavy_failed by cause: the slab the sample rays ask for overflows the shared list, */
    uint64_t heavy_failed_deferred;  /* the list of deferred nodes overflowed, */
    uint64_t heavy_failed_passes;    /* more than 128 passes */
    uint64_t heavy_cycles_walk;      /* SM clock cycles, summed over the warps of k_heavy_lists: the slab walk (of which */
    uint64_t heavy_cycles_test;      /* ... the hit tests) and */
    uint64_t heavy_cycles_publish;   /* writing the lists */
} rtgs_render_stats;

const char* rtgs_last_error(void);
int rtgs_abi_version(void);
int rtgs_device_count(int* n);

/* Scene.load_file back half — scene.py:116-160 (staging fields + build_gaussian kernel).
 * Inputs are the POST-activation parameters (scene.py:110-114): unit quaternion (x,y,z,w),
 * linear scale, sigmoid colour and opacity; `sh` is (n,15,3) float32 in the order
 * sh_10..sh_36 of gaussian.py:37-51, or NULL for SH degree 0.  Host pointers; copied. */
int rtgs_scene_create(int device, int64_t n,
                      const float* pos, const float* rot_xyzw, const float* scale,
                      const float* color, const float* opacity, const float* sh,
                      rtgs_scene** out);

/* Scene.load_file front half on the GPU — scene.py:95-114: `vertices` is the raw binary
 * little-endian PLY vertex block (n rows of `stride_floats` float32), `col` the 59 column
 * offsets in the order x,y,z, f_dc_0..2, f_rest_0..44, opacity, scale_0..2, rot_0..3 (any
 * offset < 0 = property absent -> 0).  Applies the activations of scene.py:110-114 on device.
 * sh_layout: 0 = channel-major (sh_k[c] = f_rest_{15c+k}: the 3DGS file layout, the intent of the reference's
 * reshape((-1,3,15)), scene.py:106-107), 1 = interleaved (sh_k[c] = f_rest_{3k+c}: that (N,3,15) buffer
 * reinterpreted flat as (N,15,3), which is what the Taichi stand-in behind the committed goldens executes).
 * What real Taichi stores for the reference's untransposed copy (scene.py:122,127) is not verifiable offline;
 * SURVEY.md §7 hard part 7 derives a third candidate.  The layouts are named for what they do. */
int rtgs_scene_create_from_ply_rows(int device, int64_t n, const float* vertices,
                                    int32_t stride_floats, const int32_t* col /*[59]*/,
                                    float scale, int32_t sh_layout, rtgs_scene** out);

/* BVH build — replaces scene.py:162-404 (binned-SAH host loop) with a GPU LBVH:
 * per-Gaussian preprocessing (quat -> R, W = S^-1 R^T, tight sqrt(3)-sigma AABB;
 * gaussian.py:86-138), 30-bit Morton codes, radix sort, Karras hierarchy, bottom-up refit.
 * leaf_size is accepted for Scene(leaf_prim=...) compatibility (scene.py:78-87). */
int rtgs_scene_build_bvh(rtgs_scene* s, int32_t leaf_size);
/* Device time of that build in milliseconds (CUDA events around its kernels: bounds, Morton codes, radix sort,
 * Karras, packing, refit).  The reference logs its own build time per node (scene.py:398-404). */
int rtgs_scene_build_ms(const rtgs_scene* s, float* ms);
int rtgs_scene_morton_bits(const rtgs_scene* s, int32_t* bits /* 30 or 63 */);

int rtgs_scene_num_gaussians(const rtgs_scene* s, int64_t* n);
int rtgs_scene_device(const rtgs_scene* s, int* device);

/* Parity / debug read-back of the LBVH integers (host pointers, any may be NULL):
 * morton (n) in ORIGINAL order, sorted_idx (n), child ((n-1)*2, unified ids: leaf k -> n-1+k),
 * parent (2n-1, root -1), aabb ((2n-1)*6: min xyz, max xyz). */
int rtgs_scene_read_lbvh(rtgs_scene* s, uint32_t* morton, uint32_t* sorted_idx,
                         int32_t* child, int32_t* parent, float* aabb);

/* 63-bit Morton codes (original order) of a scene built with RTGS_OPT_MORTON_BITS = 63; spec:
 * oracle/lbvh_ref.py morton63.  rtgs_scene_read_lbvh then takes morton = NULL. */
int rtgs_scene_read_morton64(rtgs_scene* s, uint64_t* codes /*n*/);

/* Read back stored Gaussian parameters in original order (Scene.gaussian_field, scene.py:131):
 * host pointers, any may be NULL.  sh is (n,15,3). */
int rtgs_scene_read_gaussians(rtgs_scene* s, float* pos, float* rot_xyzw, float* scale,
                              float* color, float* opacity, float* sh);

/* RayTracer.sample for a whole sample — ray_tracer.py:39-104 (clear_attenuation +
 * generate_ray_field + depth x sample_step) fused into one pass: camera ray generation
 * (camera.py:31-71), traversal (scene.py:406-450), intersection (gaussian.py:203-230),
 * evaluation (gaussian.py:140-201) and front-to-back compositing (ray_tracer.py:96-98) of the
 * `depth` nearest entries per pixel.
 * Region: pixels i in [x0,x0+w), j in [y0,y0+h) of the camera's (W,H) image.
 * out_rgb: device, (w,h,3) float32 i-major region buffer, or the full (W,H,3) image when
 *          `full_image_pitch` != 0 (then pixel (i,j) is written at its full-image index).
 * out_T:   device, final transmittance per pixel (attenuation_buf, ray_tracer.py:35), same
 *          indexing as out_rgb; may be NULL.
 * accumulate != 0: out_rgb += colour (sample_buf semantics, ray_tracer.py:96); else out_rgb = colour.
 * t_cut: transmittance early-termination threshold (0 disables; reference has none).
 * stats: optional host struct, filled after the stream is synchronised (forces a sync). */
int rtgs_render(rtgs_scene* s, const rtgs_camera* cam,
                int32_t x0, int32_t y0, int32_t w, int32_t h,
                int32_t depth, float t_cut, int32_t accumulate, int32_t full_image_pitch,
                float* out_rgb, float* out_T, void* stream, rtgs_render_stats* stats);

/* rtgs_render plus a depth image.  out_depth: device float32, indexed like out_T (region or full-image pitch,
 * RTGS_OPT_STRIPE stripes), ACCUMULATED (+=) with accumulate != 0 like out_rgb; NULL makes the call rtgs_render.
 * For each pixel D = sum_k T_k alpha_k t*_k over the layers the colour composites (same list, order and t_cut stop),
 * where t*_k = (p - o)^T W^T W d / |W d|^2 is the ray parameter of the point where layer k's Gaussian responds most
 * along the ray (o, d) (W = local_frame as rendered; for a hit t* > t1 > 0).  D is not normalised: the expected depth
 * is D / (1 - T).  Units are those of d: camera rays have |d| = |q_cam|^2, so for a unit camera quaternion t* is the
 * Euclidean distance from the camera centre along the ray; the camera-space z depth of pixel (i, j) is
 * t* / sqrt(px^2 + py^2 + 1) (px, py as in rtgs_render_backward_camera).  RGB and T are bit-identical to rtgs_render's,
 * and every render mode gives the same D bit for bit. */
int rtgs_render_depth(rtgs_scene* s, const rtgs_camera* cam,
                      int32_t x0, int32_t y0, int32_t w, int32_t h,
                      int32_t depth, float t_cut, int32_t accumulate, int32_t full_image_pitch,
                      float* out_rgb, float* out_T, float* out_depth, void* stream, rtgs_render_stats* stats);

/* Replace the stored parameters of a scene (same n, same SH presence) from DEVICE pointers on the scene's device
 * (layouts of rtgs_scene_create; sh NULL iff the scene has none; values must be finite), then the caller calls
 * rtgs_scene_build_bvh.  Renders/backward before the rebuild fail with RTGS_ERR_STATE.  The copies are ordered after
 * prior work on `stream`, and the rebuild (on the scene's own stream) after the copies.  The source buffers are read
 * until rtgs_scene_build_bvh returns. */
int rtgs_scene_set_gaussians_device(rtgs_scene* s, const float* pos, const float* rot_xyzw, const float* scale,
                                    const float* color, const float* opacity, const float* sh, void* stream);

/* Backward of rtgs_render for the region (x0,y0,w,h): dL_drgb (w,h,3) and optional dL_dT (w,h) are device, i-major
 * region buffers.  Gradients are ACCUMULATED (+=) into device buffers in ORIGINAL Gaussian order, layouts of
 * rtgs_scene_create (grad_sh (n,15,3)); any grad pointer may be NULL.  replay_rgb / replay_T (optional, (w,h,3)/(w,h))
 * receive the image the backward recomputed - the consistency check against rtgs_render.  Independent of
 * RTGS_OPT_RENDER_MODE / _STRIPE / _HEAVY_LISTS; uses no per-frame scene scratch.
 * The gradient is that of the image with each pixel's layer list (the `depth` nearest entries, t_cut applied) held
 * fixed: membership, order and the q = 3 silhouette have none.  The camera gets none here: see
 * rtgs_render_backward_camera. */
int rtgs_render_backward(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                         int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT,
                         float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                         float* grad_opacity, float* grad_sh, float* replay_rgb, float* replay_T, void* stream);

/* rtgs_render_backward plus the gradient with respect to the camera: grad_cam_pos (3), grad_cam_rot (4, the stored
 * x,y,z,w quaternion) and grad_cam_focal (2: fx, fy), device float32, ACCUMULATED (+=), any of them NULL.  With all
 * three NULL the call is rtgs_render_backward.  Same arguments, checks and layer-list definition otherwise.
 * The camera enters the image only through each pixel's ray: origin o = position, direction d = Rm(q) n / |n| with
 * n = (px, py, -1), px = (i + 0.5 - W/2) / fx, py = (j + 0.5 - H/2) / fy and Rm = as_rotation_mat3 of the stored
 * quaternion as given (not normalised, so |d| = |q|^2).  Per layer dq/do = 2 W^T e and dq/dd = -2 sigma W^T e (the
 * terms of the Gaussian gradient), and the SH colour depends on d / |d|.  The camera gradient is summed in float64
 * in a fixed order and rounded to float32 once per value: two identical calls give bit-identical results.  A
 * temporary buffer of 112 bytes per 4 tiles (4x8 pixels each) is allocated and freed stream-ordered on `stream`. */
int rtgs_render_backward_camera(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                                int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT,
                                float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                                float* grad_opacity, float* grad_sh,
                                float* grad_cam_pos, float* grad_cam_rot, float* grad_cam_focal,
                                float* replay_rgb, float* replay_T, void* stream);

/* rtgs_render_backward_camera plus the depth image of rtgs_render_depth: dL_dD (w,h) device or NULL, its gradient
 * flows to the Gaussians and the camera like dL_drgb's; replay_depth (w,h) or NULL receives the depth the backward
 * recomputed in float64.  With both NULL the call is rtgs_render_backward_camera (the same kernels). */
int rtgs_render_backward_depth(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                               int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT,
                               float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                               float* grad_opacity, float* grad_sh,
                               float* grad_cam_pos, float* grad_cam_rot, float* grad_cam_focal,
                               float* replay_rgb, float* replay_T, const float* dL_dD, float* replay_depth,
                               void* stream);

/* Tuning knobs of one scene's render path (no reference counterpart; defaults need no call).
 *  RTGS_OPT_RENDER_MODE      0 (default): k_tile_lists (traversal, one candidate list per 4x8-pixel tile) +
 *                            k_shade_tiles (intersection, k-buffer, compositing) + the fused kernel k_render for the
 *                            tiles whose list did not fit the pool; 2: k_frame - the same traversal and shading
 *                            code in ONE launch (persistent warps alternate between the two; lowest latency for
 *                            a single frame that is spread over four or more GPUs); 1: the fused kernel alone.
 *                            depth > 16 always uses the fused kernel.  Frames launched alternately on two streams
 *                            use separate scratch and overlap on the device in every mode.
 *  RTGS_OPT_LIST_POOL_CHUNKS capacity of the candidate-list pool in 128-byte chunks (31 candidates each);
 *                            -1 (default) = 16 chunks per 4x8-pixel tile of the rendered region, doubled whenever a
 *                            finished frame used more than 70 % of it.  A small pool is
 *                            legal (it only moves tiles to the fused kernel) and is what the tests use to
 *                            exercise that path.
 *  RTGS_OPT_KERNEL_TIMING    see rtgs_scene_read_kernel_times.
 *  RTGS_OPT_STRIPE           value = (mod << 32) | rem: following renders touch only the 32-pixel-wide column
 *                            stripes mi = (i - x0) / 32 with mi % mod == rem and leave every other pixel of the
 *                            output untouched (tile sharding of one frame over `mod` GPUs, SURVEY.md §8e; a
 *                            stripe is 32*H*3 contiguous floats of the (W,H,3) image).  (1 << 32) = all (default).
 *  RTGS_OPT_MORTON_BITS      width of the Morton codes of the NEXT rtgs_scene_build_bvh (call it again to
 *                            rebuild): 30 = the north-star spec, 63 = 21 bits per axis, 0 (default) = 30 unless
 *                            more than an eighth of the 30-bit codes repeat - far outliers, or many Gaussians
 *                            per 1/1024 of the extent - in which case the tree is rebuilt from 63-bit codes
 *                            (SURVEY.md 8f-3: BVH quality; 4 stray points among 1 M Gaussians cost the 30-bit
 *                            tree a factor 150 in frame time).  The image does not depend on the width, only
 *                            the traversal cost.  rtgs_scene_morton_bits reports the width in use. */
typedef enum rtgs_option {
    RTGS_OPT_RENDER_MODE = 0,
    RTGS_OPT_LIST_POOL_CHUNKS = 1,
    RTGS_OPT_KERNEL_TIMING = 2,
    RTGS_OPT_STRIPE = 3,
    RTGS_OPT_MORTON_BITS = 4,
    RTGS_OPT_HEAVY_LISTS = 6,    /* tiles of groups whose frustum holds more candidates than the traversal's shared-memory
                                  * list: 0 (default) = rendered by the fused kernel k_render; 1 = listed
                                  * in depth slabs by k_heavy_lists once a frame of the scene has had such groups, 2 = from
                                  * the first frame on (csrc/heavy_lists.cuh; same pixels, bit for bit).  Mode 0 renders only. */
    RTGS_OPT_HEAVY_LIMIT = 7,    /* a group is heavy above this many candidates (default -1: the capacity of the shared
                                  * list, 896; smaller values are for tests) */
    RTGS_OPT_TREE_DEPTH = 5      /* read-only: depth of the deepest LBVH leaf (root = 0); the traversal stacks are
                                  * sized for <= 96 (62 for unique 30-bit keys, 63 + 30 for repeated 63-bit codes)
                                  * and rtgs_scene_build_bvh fails with RTGS_ERR_STATE beyond that */
} rtgs_option;
int rtgs_scene_set_option(rtgs_scene* s, int32_t option, int64_t value);
/* Current value of an option (RTGS_OPT_RENDER_MODE: the mode in effect, environment default included;
 * RTGS_OPT_LIST_POOL_CHUNKS: the pool's present capacity; RTGS_OPT_MORTON_BITS: the width in use once built). */
int rtgs_scene_get_option(const rtgs_scene* s, int32_t option, int64_t* value);

/* Per-kernel device times (measurement only).  RTGS_OPT_KERNEL_TIMING = n > 0 makes every following render
 * bracket its kernels with CUDA events on the render stream (a ring of n frames; 0 switches it off).
 * rtgs_scene_read_kernel_times synchronises the device and returns, for the last `frames` renders (oldest
 * first), RTGS_NUM_KERNELS floats each, the milliseconds of the frame's (up to) three launches in order:
 * mode 0: k_tile_lists, k_shade_tiles, k_render; mode 2: 0, k_frame, k_render (the hand-over tiles); mode 1:
 * 0, 0, k_render.  Fails with RTGS_ERR_STATE if fewer frames were timed. */
#define RTGS_NUM_KERNELS 3
int rtgs_scene_read_kernel_times(rtgs_scene* s, int32_t frames, float* ms /* frames * RTGS_NUM_KERNELS */);

/* Pinned (page-locked, device-mapped) host memory for image outputs.  rtgs_render_host is
 * fastest when its output buffers come from here (DMA straight into the destination,
 * overlapped with the render); rtgs_render_host_submit requires it. */
int rtgs_host_alloc(size_t bytes, void** out);
int rtgs_host_free(void* p);

/* Peer-mapped framebuffer for tile sharding across processes (SURVEY.md 8e: "peer-mapped stores of each GPU's
 * tiles into GPU 0's framebuffer over NVLink"; no reference counterpart).  Rank 0 allocates the (W,H,3) image with
 * rtgs_device_alloc and exports it; every other rank opens the handle on its own device and passes the returned
 * pointer as `out_rgb` of rtgs_render (full_image_pitch = 1, RTGS_OPT_STRIPE set): its kernels then store their
 * stripes straight into rank 0's memory.  handle = the 64 bytes of a cudaIpcMemHandle_t. */
#define RTGS_IPC_HANDLE_BYTES 64
int rtgs_device_alloc(int device, size_t bytes, void** out);
int rtgs_device_free(int device, void* p);
int rtgs_ipc_export(int device, const void* dev_ptr, unsigned char* handle /*[64]*/);
int rtgs_ipc_open(int device, const unsigned char* handle /*[64]*/, void** out);
int rtgs_ipc_close(int device, void* p);

/* Multi-GPU hand-over without a collective (SURVEY.md 8e: "only the final framebuffer gathered, no NCCL on the hot
 * path"; ray_tracer.py:85 - pixels are independent, so ranks exchange nothing but finished pixels).  The pointers
 * are DEVICE pointers to 32-bit counters, typically in the gathering rank's memory and peer-mapped here
 * (rtgs_ipc_open).  They apply to the NEXT frame launched on the scene (rtgs_render / _render_host*) and are
 * cleared by it:
 *   arrive       when the frame's last kernel has performed all its framebuffer stores, its last CTA increments
 *                *arrive once at system scope (release).  The gathering rank waits for world x frames arrivals
 *                (rtgs_stream_wait_counter) - no extra kernel on the producing ranks, no collective.
 *   grant, grant_value   before a warp's first framebuffer store of the frame it waits until
 *                (int32)(*grant - grant_value) >= 0: the consumer has released the buffer being overwritten
 *                (rtgs_stream_set_counter on the consumer's stream); NULL = do not wait.
 * rtgs_stream_wait_counter / _set_counter queue a one-thread kernel on `stream` of `device`; _set_counter raises the
 * counter to `value` (a maximum, so that releases queued on different streams commute). */
int rtgs_scene_set_frame_sync(rtgs_scene* s, uint32_t* arrive, const uint32_t* grant, uint32_t grant_value);
int rtgs_stream_wait_counter(int device, const uint32_t* counter, uint32_t value, void* stream);
int rtgs_stream_set_counter(int device, uint32_t* counter, uint32_t value, void* stream);

/* Page-lock (and device-map) an existing host range, e.g. a POSIX shared-memory segment that several ranks
 * deliver their stripes of one frame into (each over its own PCIe link).  Portable across devices. */
int rtgs_host_register(void* p, size_t bytes);
int rtgs_host_unregister(void* p);
/* Device alias of a pinned / registered host address (for flags a stream-ordered kernel stores into host memory). */
int rtgs_host_device_pointer(void* host, void** dev);
/* Queue a one-thread kernel that release-stores `value` to *counter at system scope (a plain store: for flags in
 * mapped host memory, one writer per flag). */
int rtgs_stream_store_u32(int device, uint32_t* counter, uint32_t value, void* stream);
/* Tile sharding, host delivery: copy this rank's 32-column stripes (stripe k belongs to rank k % world, the
 * RTGS_OPT_STRIPE partition) of a (W,H,3) float32 DEVICE image to the same positions of a (W,H,3) pinned HOST image:
 * one strided DMA for all full stripes (+ one for a ragged last stripe).  With every rank delivering its own stripes
 * into one shared, registered host image the frame crosses PCIe on all the GPUs' links in parallel. */
int rtgs_copy_stripes_d2h(int device, float* host_rgb, const float* dev_rgb, int32_t W, int32_t H,
                          int32_t world, int32_t rank, void* stream);
/* The same stripes into a (W,H,3) DEVICE image, typically the gathering rank's peer-mapped frame: the bulk-copy form
 * of the gather (render into local memory, then one strided copy over NVLink) next to the default one (the render
 * kernels store into the peer frame directly).  rtgs_stream_add_counter queues a one-thread kernel that
 * release-increments *counter at system scope: the `arrive` signal of a frame gathered this way. */
int rtgs_copy_stripes_d2d(int device, float* dst_rgb, const float* dev_rgb, int32_t W, int32_t H,
                          int32_t world, int32_t rank, void* stream);
int rtgs_stream_add_counter(int device, uint32_t* counter, void* stream);

/* Same as rtgs_render but with HOST output buffers (the end-to-end call a user of
 * RayTracer makes: camera in, image out): `host_rgb` ((w,h,3) float32) and optionally
 * `host_T` ((w,h)).  Synchronous.  For pinned buffers (rtgs_host_alloc, cudaHostAlloc,
 * cudaHostRegister) the frame is rendered into device memory in up to 24 bands of 32-pixel
 * columns and every band's DMA is queued as soon as the kernels flag it complete, so the copy
 * overlaps the render; pageable buffers are staged through library-owned pinned memory. */
int rtgs_render_host(rtgs_scene* s, const rtgs_camera* cam,
                     int32_t x0, int32_t y0, int32_t w, int32_t h,
                     int32_t depth, float t_cut, float* host_rgb, float* host_T);

/* The same call split in two, for sweeps over many views (the reference's viewer loop, __main__.py:236-252,
 * and the 64-view orbit of the bench): _submit queues the frame's kernels and returns at once, _collect
 * delivers the OLDEST submitted frame to the host buffers given at its submit and returns when the image is
 * complete.  Up to two frames may be in flight, so frame f+1 renders while the last bands of frame f cross
 * PCIe.  The destination must be pinned (rtgs_host_alloc / cudaHostAlloc / cudaHostRegister) and must not
 * be touched between submit and collect.  RTGS_ERR_STATE: a third submit, a collect with nothing in
 * flight, or rtgs_render_host while frames are in flight. */
int rtgs_render_host_submit(rtgs_scene* s, const rtgs_camera* cam,
                            int32_t x0, int32_t y0, int32_t w, int32_t h,
                            int32_t depth, float t_cut, float* host_rgb, float* host_T);
int rtgs_render_host_collect(rtgs_scene* s);

/* rtgs_render_host_submit with a COMPACT host image (opt-in; the float32 call above is the parity path).  The
 * frame is rendered in float32 as always and converted on the device before the DMA:
 *   RTGS_PIXELS_F32    (w,h,3) float32, 12 B/pixel - identical to rtgs_render_host_submit
 *   RTGS_PIXELS_F16    (w,h,3) IEEE half, round to nearest even, 6 B/pixel
 *   RTGS_PIXELS_RGBA8  (w,h,4) bytes, each channel clip(x,0,1)*255 rounded to nearest, alpha 255, 4 B/pixel - what the
 *                      reference's viewer shows (ti.GUI.set_image clips to 8 bits, __main__.py:249-252)
 * For viewer loops and sweeps on several GPUs of one host, whose summed device-to-host traffic otherwise exceeds
 * what the host can absorb (profiles/README.md: ~100 GB/s in total on the 8-GPU box).  Collected with
 * rtgs_render_host_collect like any submitted frame. */
typedef enum rtgs_pixel_format { RTGS_PIXELS_F32 = 0, RTGS_PIXELS_F16 = 1, RTGS_PIXELS_RGBA8 = 2 } rtgs_pixel_format;
int rtgs_render_host_submit_packed(rtgs_scene* s, const rtgs_camera* cam,
                                   int32_t x0, int32_t y0, int32_t w, int32_t h,
                                   int32_t depth, float t_cut, void* host_pixels, int32_t format);

/* Camera.generate_ray_field — camera.py:57-71.  rays: device, (W,H,8) float32
 * = origin xyz, direction xyz, start, end (ray.py:4-18). */
int rtgs_generate_rays(const rtgs_camera* cam, int device, float* rays, void* stream);

/* Scene.hit for a batch of rays — scene.py:406-450: per ray the Gaussian with the smallest
 * entry distance t1 in (start, end).  rays: device (n,8) as above.  idx: device int32 (n)
 * = ORIGINAL Gaussian index or -1; t12: device (n,2) float32 (+inf on a miss). */
int rtgs_trace_closest(rtgs_scene* s, int64_t nrays, const float* rays,
                       int32_t* idx, float* t12, void* stream);

/* Render arbitrary rays: non-pinhole cameras, ray batches drawn from many views, secondary rays.  rays: device
 * (nrays,8) float32 as above, 16-byte aligned: origin o, direction d (used as given, not normalised; the SH colour
 * uses d / |d|), start, end.  A ray's layer list is the Gaussians whose float64 exact intersection has
 * start < t1 < end, in ascending t1 (exact ties by sorted position), truncated to `depth`, composited front to back
 * while the incoming float32 T >= t_cut.  start = 0, end = +inf is the pixel rule of rtgs_render, so a ray of
 * rtgs_generate_rays gives its pixel's layer list (up to the float32 rounding of d).  A ray with a non-finite o or d
 * component, d = 0 or !(start < end) composites nothing: rgb 0, T 1.
 * out_rgb: device (nrays,3); out_T: device (nrays) or NULL.  Stream-ordered on `stream`, no scene scratch.
 * nrays = 0 does nothing. */
int rtgs_render_rays(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                     float* out_rgb, float* out_T, void* stream);

/* rtgs_render_rays plus out_depth (nrays) device or NULL (then the call is rtgs_render_rays): D of rtgs_render_depth
 * for each ray, t* in units of the ray's own d, float64 per ray.  A t* may lie beyond the ray's `end`; a degenerate
 * ray gets D = 0.  RGB and T are bit-identical to rtgs_render_rays's. */
int rtgs_render_rays_depth(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                           float* out_rgb, float* out_T, float* out_depth, void* stream);

/* Backward of rtgs_render_rays with each ray's layer list and t_cut stop held fixed (the definition of
 * rtgs_render_backward).  dL_drgb (nrays,3) and dL_dT (nrays, or NULL) are device buffers.  The Gaussian gradients
 * are ACCUMULATED as in rtgs_render_backward (any may be NULL).  grad_rays (nrays,8) or NULL is ACCUMULATED too:
 * columns 0-2 dL/do, 3-5 dL/dd, 6-7 untouched (start, end and depth have no gradient); each ray's thread adds its own
 * values, so two identical calls give bit-identical ray gradients.  Degenerate rays get no gradient.  replay_rgb /
 * replay_T (optional) receive the image recomputed, bit-identical to rtgs_render_rays. */
int rtgs_render_rays_backward(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                              const float* dL_drgb, const float* dL_dT,
                              float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                              float* grad_opacity, float* grad_sh, float* grad_rays,
                              float* replay_rgb, float* replay_T, void* stream);

/* rtgs_render_rays_backward plus dL_dD (nrays) device or NULL, the gradient of rtgs_render_rays_depth's depth, which
 * flows to the Gaussians and to grad_rays like dL_drgb's, and replay_depth (nrays) or NULL, bit-identical to
 * rtgs_render_rays_depth's out_depth.  With both NULL the call is rtgs_render_rays_backward (the same kernels). */
int rtgs_render_rays_backward_depth(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                                    const float* dL_drgb, const float* dL_dT,
                                    float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                                    float* grad_opacity, float* grad_sh, float* grad_rays,
                                    float* replay_rgb, float* replay_T, const float* dL_dD, float* replay_depth,
                                    void* stream);

int rtgs_scene_destroy(rtgs_scene* s);

#ifdef __cplusplus
}
#endif
#endif /* RTGS_B200_H */
