// abi.cu — extern "C" boundary (include/rtgs_b200.h): scene lifetime, build, render, read-back.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <cmath>
#include <new>

#include "render_common.cuh"

static thread_local char g_err[512] = "";

void rtgs_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

template <typename T>
int dev_alloc(T** p, size_t count) {
    *p = nullptr;
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
    if (e != cudaSuccess) {
        rtgs_set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? RTGS_ERR_NOMEM : RTGS_ERR_CUDA;
    }
    return RTGS_OK;
}

void free_scene(rtgs_scene* s) {
    if (!s) return;
    DeviceGuard g(s->device);
    cudaFree(s->pos); cudaFree(s->rot); cudaFree(s->scale); cudaFree(s->color); cudaFree(s->opacity);
    cudaFree(s->sh); cudaFree(s->morton); cudaFree(s->sorted_idx); cudaFree(s->child); cudaFree(s->parent);
    cudaFree(s->morton64);
    if (s->shp_tex) cudaDestroyTextureObject(s->shp_tex);
    cudaFree(s->aabb); cudaFree(s->geo); cudaFree(s->shp); cudaFree(s->raw); cudaFree(s->nodes); cudaFree(s->leafbox); cudaFree(s->nodes4);
    for (auto& fs : s->scratch) {
        cudaFree(fs.tile_desc); cudaFree(fs.list_pool); cudaFree(fs.fallback_tiles); cudaFree(fs.fallback_tiles2); cudaFree(fs.ready);
        cudaFree(fs.heavy_groups); cudaFree(fs.tile_cap); cudaFree(fs.heavy_scratch);
        cudaFree(fs.counters);
        if (fs.free_event) cudaEventDestroy(fs.free_event);
    }
    cudaFree(s->stats_dev);
    for (auto& hs : s->host_slot) {
        cudaFree(hs.stage_rgb); cudaFree(hs.stage_T); cudaFree(hs.stage_packed);
        if (hs.done) cudaEventDestroy(hs.done);
        if (hs.copied) cudaEventDestroy(hs.copied);
    }
    if (s->pinned_rgb) cudaFreeHost(s->pinned_rgb);
    if (s->pinned_T) cudaFreeHost(s->pinned_T);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    if (s->own_stream2) cudaStreamDestroy(s->own_stream2);
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    if (s->copy_stream2) cudaStreamDestroy(s->copy_stream2);
    cudaFree(s->band_done);
    if (s->band_flags) cudaFreeHost(s->band_flags);
    for (cudaEvent_t e : s->timing_events) cudaEventDestroy(e);
    delete s;
}

#define TRY(expr)                      \
    do {                               \
        int _r = (expr);               \
        if (_r != RTGS_OK) return _r;  \
    } while (0)

int alloc_scene(int device, int64_t n, bool has_sh, rtgs_scene** out) {
    rtgs_scene* s = new (std::nothrow) rtgs_scene();
    if (!s) {
        rtgs_set_error("out of host memory");
        return RTGS_ERR_NOMEM;
    }
    s->device = device;
    s->n = n;
    s->has_sh = has_sh;
    s->num_nodes = n > 1 ? n - 1 : 1;
    *out = s;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    s->sm_count = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s->own_stream2, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s->copy_stream2, cudaStreamNonBlocking));
    // [0, MAX) band flags of host slot 0, [MAX, 2 MAX) those of host slot 1, then four mirror words per frame scratch
    CUDA_TRY(cudaHostAlloc((void**)&s->band_flags, (2 * RTGS_MAX_BANDS + 8) * sizeof(int), cudaHostAllocMapped));
    CUDA_TRY(cudaHostGetDevicePointer((void**)&s->band_flags_dev, s->band_flags, 0));
    for (int k = 0; k < 2; ++k) {
        const int off = k * RTGS_MAX_BANDS;
        s->host_slot[k].flags = s->band_flags + off;
        s->host_slot[k].flags_dev = s->band_flags_dev + off;
        CUDA_TRY(cudaEventCreateWithFlags(&s->host_slot[k].done, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&s->host_slot[k].copied, cudaEventDisableTiming));
    }
    TRY(dev_alloc(&s->band_done, RTGS_MAX_BANDS));
    for (int k = 0; k < 2; ++k) {
        rtgs_scene::FrameScratch& fs = s->scratch[k];
        const int off = 2 * RTGS_MAX_BANDS + 4 * k;
        fs.mirror = s->band_flags + off;
        fs.mirror_dev = s->band_flags_dev + off;
        fs.mirror[0] = 0;   // pool demand of the last finished frame (render.cu: ensure_lists)
        fs.mirror[1] = 0;   // some finished frame had fallback tiles (render.cu: launch_render_k)
        fs.mirror[2] = 0;   // some frame had groups whose candidate list overflows shared memory (render.cu: k_heavy_lists)
        fs.mirror[3] = 0;
        TRY(dev_alloc(&fs.counters, 16));      // CTR_COUNT (render_common.cuh)
        CUDA_TRY(cudaMemset(fs.counters, 0, 16 * sizeof(unsigned int)));   // k_frame leaves them zeroed frame after frame
        CUDA_TRY(cudaEventCreateWithFlags(&fs.free_event, cudaEventDisableTiming));
    }
    TRY(dev_alloc(&s->pos, n * 3));
    TRY(dev_alloc(&s->rot, n * 4));
    TRY(dev_alloc(&s->scale, n * 3));
    TRY(dev_alloc(&s->color, n * 3));
    TRY(dev_alloc(&s->opacity, n));
    if (has_sh) TRY(dev_alloc(&s->sh, n * 45));
    TRY(dev_alloc(&s->morton, n));
    TRY(dev_alloc(&s->sorted_idx, n));
    TRY(dev_alloc(&s->child, (n > 1 ? n - 1 : 1) * 2));
    TRY(dev_alloc(&s->parent, 2 * n - 1));
    TRY(dev_alloc(&s->aabb, (2 * n - 1) * 6));
    TRY(dev_alloc(&s->geo, n * 4));
    if (has_sh) {
        // the SH records and a linear float4 texture over them (eval_colour fetches part of a record through the
        // texture path: the LSU pipe bounds the shading, the TEX pipe has throughput to spare).  Scenes too large for
        // one linear texture get no texture and eval_colour loads the whole record.
        TRY(dev_alloc(&s->shp, n * 12));
        const char* tex_env = getenv("RTGS_SH_TEX");     // "0": no texture, loads only (what huge scenes get; tests)
        const bool tex_off = tex_env != nullptr && atoi(tex_env) == 0;
        if (!tex_off && n <= rtgs_dev::SH_TEX_MAX_RECORDS) {
            cudaResourceDesc rd = {};
            rd.resType = cudaResourceTypeLinear;
            rd.res.linear.devPtr = s->shp;
            rd.res.linear.desc = cudaCreateChannelDesc<float4>();
            rd.res.linear.sizeInBytes = (size_t)n * 12 * sizeof(float4);
            cudaTextureDesc td = {};
            td.readMode = cudaReadModeElementType;
            CUDA_TRY(cudaCreateTextureObject(&s->shp_tex, &rd, &td, nullptr));
        }
    }
    TRY(dev_alloc(&s->raw, n * 3));
    TRY(dev_alloc(&s->nodes, s->num_nodes * 4));
    TRY(dev_alloc(&s->leafbox, n * 2));
    TRY(dev_alloc(&s->nodes4, s->num_nodes * 8));
    TRY(dev_alloc(&s->stats_dev, 32));   // ST_TOTAL (render_common.cuh)
    return RTGS_OK;
}

int ensure_stage(rtgs_scene::HostSlot& hs, size_t pixels) {
    if (hs.stage_pixels < pixels) {
        cudaFree(hs.stage_rgb);   // (synchronises with the device: no frame is reading it any more)
        cudaFree(hs.stage_T);
        hs.stage_rgb = hs.stage_T = nullptr;
        hs.stage_pixels = 0;
        TRY(dev_alloc(&hs.stage_rgb, pixels * 3));
        TRY(dev_alloc(&hs.stage_T, pixels));
        hs.stage_pixels = pixels;
    }
    return RTGS_OK;
}

int ensure_pinned(rtgs_scene* s, size_t pixels) {
    if (s->pinned_pixels < pixels) {
        if (s->pinned_rgb) cudaFreeHost(s->pinned_rgb);
        if (s->pinned_T) cudaFreeHost(s->pinned_T);
        s->pinned_rgb = s->pinned_T = nullptr;
        s->pinned_pixels = 0;
        CUDA_TRY(cudaMallocHost((void**)&s->pinned_rgb, pixels * 3 * sizeof(float)));
        CUDA_TRY(cudaMallocHost((void**)&s->pinned_T, pixels * sizeof(float)));
        s->pinned_pixels = pixels;
    }
    return RTGS_OK;
}

bool all_finite(const float* v, int64_t count) {
    bool fin = true;
    for (int64_t i = 0; i < count; ++i) fin = fin && std::isfinite(v[i]);
    return fin;
}

int check_camera(const rtgs_camera* cam) {
    RTGS_CHECK_ARG(cam != nullptr);
    RTGS_CHECK_ARG(cam->width > 0 && cam->height > 0);
    RTGS_CHECK_ARG(cam->focal[0] != 0.0f && cam->focal[1] != 0.0f);
    return RTGS_OK;
}

bool aligned(const void* p, uintptr_t bytes) { return ((uintptr_t)p & (bytes - 1)) == 0; }

// The checks both ray entry points share: everything but the state of the scene, before any CUDA call.
int check_rays(const rtgs_scene* s, int64_t nrays, const float* rays, const float* rgb, int32_t depth,
                      float t_cut) {
    RTGS_CHECK_ARG(s != nullptr);
    RTGS_CHECK_ARG(nrays >= 0);
    RTGS_CHECK_ARG(nrays == 0 || (rays != nullptr && aligned(rays, 16)));
    RTGS_CHECK_ARG(nrays == 0 || (rgb != nullptr && aligned(rgb, 4)));
    RTGS_CHECK_ARG(depth >= 1 && depth <= RTGS_MAX_DEPTH);
    RTGS_CHECK_ARG(t_cut >= 0.0f && t_cut < 1.0f);
    return RTGS_OK;
}

}  // namespace

extern "C" {

const char* rtgs_last_error(void) { return g_err; }
int rtgs_abi_version(void) { return RTGS_ABI_VERSION; }

int rtgs_device_count(int* n) {
    RTGS_CHECK_ARG(n != nullptr);
    CUDA_TRY(cudaGetDeviceCount(n));
    return RTGS_OK;
}

int rtgs_scene_create(int device, int64_t n, const float* pos, const float* rot_xyzw, const float* scale,
                      const float* color, const float* opacity, const float* sh, rtgs_scene** out) {
    RTGS_CHECK_ARG(out != nullptr);
    *out = nullptr;
    RTGS_CHECK_ARG(n >= 1 && n < (1ll << 30));
    RTGS_CHECK_ARG(pos && rot_xyzw && scale && color && opacity);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    // Morton codes, the hierarchy and every box test assume finite geometry: a NaN / Inf centre, rotation or scale
    // has no place in the tree (and the reference's own SAH split would not survive it either: scene.py:263-266)
    if (!all_finite(pos, n * 3) || !all_finite(rot_xyzw, n * 4) || !all_finite(scale, n * 3)) {
        rtgs_set_error("rtgs_scene_create: positions, rotations and scales must be finite (NaN or Inf found)");
        return RTGS_ERR_INVALID;
    }
    rtgs_scene* s = nullptr;
    int r = alloc_scene(device, n, sh != nullptr, &s);
    if (r == RTGS_OK) {
        // uploads are queued on the stream the build runs on (a pageable cudaMemcpy on the legacy stream is not
        // ordered against a non-blocking stream); the host arrays are borrowed only until this call returns
        cudaStream_t st = s->own_stream;
        auto up = [&](float* d, const float* h, size_t cnt) {
            return cudaMemcpyAsync(d, h, cnt * sizeof(float), cudaMemcpyHostToDevice, st) == cudaSuccess;
        };
        bool ok = up(s->pos, pos, n * 3) && up(s->rot, rot_xyzw, n * 4) && up(s->scale, scale, n * 3) &&
                  up(s->color, color, n * 3) && up(s->opacity, opacity, n) && (!sh || up(s->sh, sh, n * 45));
        ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
        if (!ok) {
            rtgs_set_error("host->device upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            r = RTGS_ERR_CUDA;
        }
    }
    if (r != RTGS_OK) {
        free_scene(s);
        return r;
    }
    *out = s;
    return RTGS_OK;
}

int rtgs_scene_create_from_ply_rows(int device, int64_t n, const float* vertices, int32_t stride_floats,
                                    const int32_t* col, float scale, int32_t sh_layout, rtgs_scene** out) {
    RTGS_CHECK_ARG(out != nullptr);
    *out = nullptr;
    RTGS_CHECK_ARG(n >= 1 && n < (1ll << 30));
    RTGS_CHECK_ARG(vertices && col && stride_floats > 0);
    RTGS_CHECK_ARG(sh_layout == 0 || sh_layout == 1);
    bool has_sh = false;
    for (int k = 6; k < 51; ++k) has_sh = has_sh || col[k] >= 0;
    for (int k = 0; k < 59; ++k) RTGS_CHECK_ARG(col[k] < stride_floats);
    // finite geometry only (see rtgs_scene_create): x,y,z (0-2), log-scales (52-54), rot_0..3 (55-58)
    for (int64_t i = 0; i < n; ++i) {
        const float* row = vertices + i * stride_floats;
        bool fin = true;
        for (int k : {0, 1, 2, 52, 53, 54, 55, 56, 57, 58})
            if (col[k] >= 0) fin = fin && std::isfinite(row[col[k]]);
        if (!fin) {
            rtgs_set_error("rtgs_scene_create_from_ply_rows: vertex %lld has a NaN or Inf position, scale or rotation",
                           (long long)i);
            return RTGS_ERR_INVALID;
        }
    }
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    rtgs_scene* s = nullptr;
    int r = alloc_scene(device, n, has_sh, &s);
    float* rows = nullptr;
    int32_t* dcol = nullptr;
    if (r == RTGS_OK) r = dev_alloc(&rows, (size_t)n * stride_floats);
    if (r == RTGS_OK) r = dev_alloc(&dcol, 59);
    if (r == RTGS_OK) {
        cudaStream_t st = s->own_stream;   // same stream as the activation kernel and the build
        cudaError_t e = cudaMemcpyAsync(rows, vertices, (size_t)n * stride_floats * sizeof(float),
                                        cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dcol, col, 59 * sizeof(int32_t), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            rtgs_set_error("host->device upload failed: %s", cudaGetErrorString(e));
            r = RTGS_ERR_CUDA;
        }
    }
    if (r == RTGS_OK)
        r = rtgs_launch_activate_ply(n, rows, stride_floats, dcol, scale, sh_layout, s->pos, s->rot, s->scale,
                                     s->color, s->opacity, s->sh, s->own_stream);
    if (r == RTGS_OK && cudaStreamSynchronize(s->own_stream) != cudaSuccess) {
        rtgs_set_error("activation kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
        r = RTGS_ERR_CUDA;
    }
    cudaFree(rows);
    cudaFree(dcol);
    if (r != RTGS_OK) {
        free_scene(s);
        return r;
    }
    *out = s;
    return RTGS_OK;
}

int rtgs_scene_build_bvh(rtgs_scene* s, int32_t leaf_size) {
    RTGS_CHECK_ARG(s != nullptr);
    (void)leaf_size;  // LBVH leaves hold one Gaussian; accepted for Scene(leaf_prim=...) compatibility
    DeviceGuard g(s->device);
    s->built = false;
    s->morton_bits_used = s->opt_morton_bits == 63 ? 63 : 30;
    int r = rtgs_lbvh_build(s);
    // automatic width: the 30-bit tree is the specification; it is replaced by the 63-bit one when more than an
    // eighth of the codes repeat, i.e. when 10 bits per axis do not resolve the scene (far outliers, or many
    // Gaussians per 1/1024 of the extent), which is when its traversal cost explodes
    if (r == RTGS_OK && s->opt_morton_bits == 0 && s->distinct_codes >= 0 && s->distinct_codes * 8 < s->n * 7) {
        const float first_ms = s->build_ms;
        s->morton_bits_used = 63;
        r = rtgs_lbvh_build(s);
        s->build_ms += first_ms;
    }
    if (r == RTGS_OK) s->built = true;
    return r;
}

int rtgs_scene_morton_bits(const rtgs_scene* s, int32_t* bits) {
    RTGS_CHECK_ARG(s != nullptr && bits != nullptr);
    if (!s->built) {
        rtgs_set_error("rtgs_scene_morton_bits: call rtgs_scene_build_bvh first");
        return RTGS_ERR_STATE;
    }
    *bits = s->morton_bits_used;
    return RTGS_OK;
}

int rtgs_scene_build_ms(const rtgs_scene* s, float* ms) {
    RTGS_CHECK_ARG(s != nullptr && ms != nullptr);
    if (!s->built) {
        rtgs_set_error("rtgs_scene_build_ms: call rtgs_scene_build_bvh first");
        return RTGS_ERR_STATE;
    }
    *ms = s->build_ms;
    return RTGS_OK;
}

int rtgs_scene_num_gaussians(const rtgs_scene* s, int64_t* n) {
    RTGS_CHECK_ARG(s && n);
    *n = s->n;
    return RTGS_OK;
}

int rtgs_scene_device(const rtgs_scene* s, int* device) {
    RTGS_CHECK_ARG(s && device);
    *device = s->device;
    return RTGS_OK;
}

int rtgs_scene_read_lbvh(rtgs_scene* s, uint32_t* morton, uint32_t* sorted_idx, int32_t* child, int32_t* parent,
                         float* aabb) {
    RTGS_CHECK_ARG(s != nullptr);
    if (!s->built) {
        rtgs_set_error("rtgs_scene_read_lbvh: BVH not built");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    const int64_t n = s->n;
    if (morton && s->morton_bits_used == 63) {
        rtgs_set_error("rtgs_scene_read_lbvh: the scene was built with 63-bit codes; read them with "
                       "rtgs_scene_read_morton64 and pass morton = NULL here");
        return RTGS_ERR_STATE;
    }
    if (morton) CUDA_TRY(cudaMemcpy(morton, s->morton, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (sorted_idx) CUDA_TRY(cudaMemcpy(sorted_idx, s->sorted_idx, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (child && n > 1) CUDA_TRY(cudaMemcpy(child, s->child, (n - 1) * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (parent) CUDA_TRY(cudaMemcpy(parent, s->parent, (2 * n - 1) * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (aabb) CUDA_TRY(cudaMemcpy(aabb, s->aabb, (2 * n - 1) * 6 * sizeof(float), cudaMemcpyDeviceToHost));
    return RTGS_OK;
}

int rtgs_scene_read_morton64(rtgs_scene* s, uint64_t* codes) {
    RTGS_CHECK_ARG(s != nullptr && codes != nullptr);
    if (!s->built || s->morton_bits_used != 63 || !s->morton64) {
        rtgs_set_error("rtgs_scene_read_morton64: the BVH was not built with RTGS_OPT_MORTON_BITS = 63");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    CUDA_TRY(cudaMemcpy(codes, s->morton64, s->n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return RTGS_OK;
}

int rtgs_scene_read_gaussians(rtgs_scene* s, float* pos, float* rot_xyzw, float* scale, float* color,
                              float* opacity, float* sh) {
    RTGS_CHECK_ARG(s != nullptr);
    DeviceGuard g(s->device);
    const int64_t n = s->n;
    if (pos) CUDA_TRY(cudaMemcpy(pos, s->pos, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    if (rot_xyzw) CUDA_TRY(cudaMemcpy(rot_xyzw, s->rot, n * 4 * sizeof(float), cudaMemcpyDeviceToHost));
    if (scale) CUDA_TRY(cudaMemcpy(scale, s->scale, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    if (color) CUDA_TRY(cudaMemcpy(color, s->color, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    if (opacity) CUDA_TRY(cudaMemcpy(opacity, s->opacity, n * sizeof(float), cudaMemcpyDeviceToHost));
    if (sh) {
        if (s->has_sh) CUDA_TRY(cudaMemcpy(sh, s->sh, n * 45 * sizeof(float), cudaMemcpyDeviceToHost));
        else memset(sh, 0, n * 45 * sizeof(float));
    }
    return RTGS_OK;
}

int rtgs_render(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h, int32_t depth,
                float t_cut, int32_t accumulate, int32_t full_image_pitch, float* out_rgb, float* out_T, void* stream,
                rtgs_render_stats* stats) {
    return rtgs_render_depth(s, cam, x0, y0, w, h, depth, t_cut, accumulate, full_image_pitch, out_rgb, out_T, nullptr,
                             stream, stats);
}

int rtgs_render_depth(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                      int32_t depth, float t_cut, int32_t accumulate, int32_t full_image_pitch, float* out_rgb,
                      float* out_T, float* out_depth, void* stream, rtgs_render_stats* stats) {
    RTGS_CHECK_ARG(s != nullptr);
    TRY(check_camera(cam));
    RTGS_CHECK_ARG(out_rgb != nullptr);
    RTGS_CHECK_ARG(aligned(out_depth, 4));
    RTGS_CHECK_ARG(w > 0 && h > 0 && x0 >= 0 && y0 >= 0 && x0 + w <= cam->width && y0 + h <= cam->height);
    RTGS_CHECK_ARG(depth >= 1 && depth <= RTGS_MAX_DEPTH);
    RTGS_CHECK_ARG(t_cut >= 0.0f && t_cut < 1.0f);
    if (!s->built) {
        rtgs_set_error("%s: call rtgs_scene_build_bvh first", out_depth ? "rtgs_render_depth" : "rtgs_render");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    cudaStream_t st = (cudaStream_t)stream;
    TRY(rtgs_launch_render(s, cam, x0, y0, w, h, depth, t_cut, accumulate, full_image_pitch, out_rgb, out_T, out_depth,
                           st, stats != nullptr));
    if (stats) {
        unsigned long long hs[32];
        CUDA_TRY(cudaMemcpyAsync(hs, s->stats_dev, sizeof(hs), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        stats->rays = hs[0]; stats->rays_hit = hs[1]; stats->layers = hs[2]; stats->nodes_tested = hs[3];
        stats->candidates = hs[4]; stats->pair_tests = hs[5]; stats->f64_refinements = hs[6]; stats->tiles = hs[7];
        stats->traversal_steps = hs[8]; stats->insert_rounds = hs[9]; stats->fallback_tiles = hs[10]; stats->useful_candidates = hs[11];
        stats->max_lists_stack = hs[12]; stats->max_fused_stack = hs[13]; stats->max_group_list = hs[14];
        stats->heavy_groups = hs[15]; stats->heavy_failed = hs[16]; stats->heavy_passes = hs[17];
        stats->heavy_sample_tests = hs[18]; stats->max_deferred = hs[19]; stats->heavy_retries = hs[20];
        stats->heavy_cycles_walk = hs[24]; stats->heavy_cycles_test = hs[25]; stats->heavy_cycles_publish = hs[26];
        stats->heavy_failed_list = hs[21]; stats->heavy_failed_deferred = hs[22]; stats->heavy_failed_passes = hs[23];
    }
    return RTGS_OK;
}

int rtgs_scene_set_gaussians_device(rtgs_scene* s, const float* pos, const float* rot_xyzw, const float* scale,
                                    const float* color, const float* opacity, const float* sh, void* stream) {
    RTGS_CHECK_ARG(s != nullptr);
    RTGS_CHECK_ARG(pos && rot_xyzw && scale && color && opacity);
    RTGS_CHECK_ARG((sh != nullptr) == s->has_sh);
    DeviceGuard g(s->device);
    cudaStream_t st = (cudaStream_t)stream;
    // renders and backward passes read the packed records, which only the rebuild refreshes
    s->built = false;
    const int64_t n = s->n;
    auto cp = [&](float* d, const float* src, size_t cnt) {
        return cudaMemcpyAsync(d, src, cnt * sizeof(float), cudaMemcpyDeviceToDevice, st);
    };
    CUDA_TRY(cp(s->pos, pos, n * 3));
    CUDA_TRY(cp(s->rot, rot_xyzw, n * 4));
    CUDA_TRY(cp(s->scale, scale, n * 3));
    CUDA_TRY(cp(s->color, color, n * 3));
    CUDA_TRY(cp(s->opacity, opacity, n));
    if (sh) CUDA_TRY(cp(s->sh, sh, n * 45));
    // the build runs on the scene's own stream: it starts after the copies (and everything before them on `stream`,
    // e.g. a backward pass still reading the old records)
    cudaEvent_t ev = nullptr;
    CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t e = cudaEventRecord(ev, st);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(s->own_stream, ev, 0);
    cudaEventDestroy(ev);
    CUDA_TRY(e);
    return RTGS_OK;
}

static int render_backward(const char* name, rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0,
                           int32_t w, int32_t h, int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT,
                           const float* dL_dD, float* const grads[6], float* const cam_grads[3], float* replay_rgb,
                           float* replay_T, float* replay_depth, void* stream) {
    RTGS_CHECK_ARG(s != nullptr);
    TRY(check_camera(cam));
    RTGS_CHECK_ARG(dL_drgb != nullptr);
    RTGS_CHECK_ARG(aligned(dL_dD, 4) && aligned(replay_depth, 4));
    RTGS_CHECK_ARG(w > 0 && h > 0 && x0 >= 0 && y0 >= 0 && x0 + w <= cam->width && y0 + h <= cam->height);
    RTGS_CHECK_ARG(depth >= 1 && depth <= RTGS_MAX_DEPTH);
    RTGS_CHECK_ARG(t_cut >= 0.0f && t_cut < 1.0f);
    if (!s->built) {
        rtgs_set_error("%s: call rtgs_scene_build_bvh first", name);
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    return rtgs_launch_render_backward(s, cam, x0, y0, w, h, depth, t_cut, dL_drgb, dL_dT, dL_dD, grads, cam_grads,
                                       replay_rgb, replay_T, replay_depth, (cudaStream_t)stream);
}

int rtgs_render_backward(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                         int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT, float* grad_pos,
                         float* grad_rot, float* grad_scale, float* grad_color, float* grad_opacity, float* grad_sh,
                         float* replay_rgb, float* replay_T, void* stream) {
    float* const grads[6] = {grad_pos, grad_rot, grad_scale, grad_color, grad_opacity, grad_sh};
    float* const cam_grads[3] = {nullptr, nullptr, nullptr};
    return render_backward("rtgs_render_backward", s, cam, x0, y0, w, h, depth, t_cut, dL_drgb, dL_dT, nullptr, grads,
                           cam_grads, replay_rgb, replay_T, nullptr, stream);
}

int rtgs_render_backward_camera(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                                int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT,
                                float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                                float* grad_opacity, float* grad_sh, float* grad_cam_pos, float* grad_cam_rot,
                                float* grad_cam_focal, float* replay_rgb, float* replay_T, void* stream) {
    return rtgs_render_backward_depth(s, cam, x0, y0, w, h, depth, t_cut, dL_drgb, dL_dT, grad_pos, grad_rot,
                                      grad_scale, grad_color, grad_opacity, grad_sh, grad_cam_pos, grad_cam_rot,
                                      grad_cam_focal, replay_rgb, replay_T, nullptr, nullptr, stream);
}

int rtgs_render_backward_depth(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                               int32_t depth, float t_cut, const float* dL_drgb, const float* dL_dT,
                               float* grad_pos, float* grad_rot, float* grad_scale, float* grad_color,
                               float* grad_opacity, float* grad_sh, float* grad_cam_pos, float* grad_cam_rot,
                               float* grad_cam_focal, float* replay_rgb, float* replay_T, const float* dL_dD,
                               float* replay_depth, void* stream) {
    float* const grads[6] = {grad_pos, grad_rot, grad_scale, grad_color, grad_opacity, grad_sh};
    float* const cam_grads[3] = {grad_cam_pos, grad_cam_rot, grad_cam_focal};
    const bool with_depth = dL_dD != nullptr || replay_depth != nullptr;
    return render_backward(with_depth ? "rtgs_render_backward_depth" : "rtgs_render_backward_camera", s, cam, x0, y0,
                           w, h, depth, t_cut, dL_drgb, dL_dT, dL_dD, grads, cam_grads, replay_rgb, replay_T,
                           replay_depth, stream);
}

int rtgs_scene_set_option(rtgs_scene* s, int32_t option, int64_t value) {
    RTGS_CHECK_ARG(s != nullptr);
    switch (option) {
        case RTGS_OPT_RENDER_MODE:
            RTGS_CHECK_ARG(value >= 0 && value <= 2);
            s->opt_render_mode = (int)value;
            return RTGS_OK;
        case RTGS_OPT_LIST_POOL_CHUNKS: {
            RTGS_CHECK_ARG(value >= -1 && value <= (1ll << 26));
            DeviceGuard g(s->device);
            s->opt_pool_chunks = value;
            // dropped here, re-created with the new capacity by the next render
            for (auto& fs : s->scratch) {
                cudaFree(fs.tile_desc); cudaFree(fs.list_pool); cudaFree(fs.fallback_tiles); cudaFree(fs.fallback_tiles2); cudaFree(fs.ready);
                cudaFree(fs.heavy_groups); cudaFree(fs.tile_cap);
                fs.heavy_groups = nullptr; fs.tile_cap = nullptr;
                fs.tile_desc = nullptr; fs.list_pool = nullptr; fs.fallback_tiles = nullptr; fs.fallback_tiles2 = nullptr; fs.ready = nullptr;
                fs.list_tiles = 0;
                fs.pool_chunks = 0;
            }
            return RTGS_OK;
        }
        case RTGS_OPT_MORTON_BITS:
            RTGS_CHECK_ARG(value == 0 || value == 30 || value == 63);
            s->opt_morton_bits = (int)value;   // takes effect at the next rtgs_scene_build_bvh
            return RTGS_OK;
        case RTGS_OPT_STRIPE: {
            const int64_t mod = value >> 32, rem = value & 0xffffffffll;
            RTGS_CHECK_ARG(mod >= 1 && mod <= 1024 && rem >= 0 && rem < mod);
            s->opt_stripe_mod = (int)mod;
            s->opt_stripe_rem = (int)rem;
            return RTGS_OK;
        }
        case RTGS_OPT_KERNEL_TIMING: {
            RTGS_CHECK_ARG(value >= 0 && value <= 4096);
            DeviceGuard g(s->device);
            CUDA_TRY(cudaDeviceSynchronize());
            for (cudaEvent_t e : s->timing_events) cudaEventDestroy(e);
            s->timing_events.clear();
            s->timing_ran.assign((size_t)value, 0);
            s->timing_frames = 0;
            for (int64_t k = 0; k < value * 4; ++k) {
                cudaEvent_t e;
                CUDA_TRY(cudaEventCreate(&e));
                s->timing_events.push_back(e);
            }
            return RTGS_OK;
        }
        case RTGS_OPT_HEAVY_LISTS:
            RTGS_CHECK_ARG(value >= -1 && value <= 2);
            s->opt_heavy_lists = (int)value;
            return RTGS_OK;
        case RTGS_OPT_HEAVY_LIMIT:
            RTGS_CHECK_ARG(value >= -1 && value <= (1ll << 30));
            s->opt_heavy_limit = (int)value;
            return RTGS_OK;
        case RTGS_OPT_TREE_DEPTH:
            rtgs_set_error("RTGS_OPT_TREE_DEPTH is read-only");
            return RTGS_ERR_INVALID;
        default:
            rtgs_set_error("unknown option %d", (int)option);
            return RTGS_ERR_INVALID;
    }
}

int rtgs_scene_get_option(const rtgs_scene* s, int32_t option, int64_t* value) {
    RTGS_CHECK_ARG(s != nullptr && value != nullptr);
    switch (option) {
        case RTGS_OPT_RENDER_MODE: {
            // the mode a depth <= 16 frame renders in: the per-scene option, else RTGS_RENDER_MODE, else 0
            int m = s->opt_render_mode;
            if (m < 0) {
                const char* e = getenv("RTGS_RENDER_MODE");
                m = e ? atoi(e) : 0;
                if (m < 0 || m > 2) m = 0;
            }
            *value = m;
            return RTGS_OK;
        }
        case RTGS_OPT_LIST_POOL_CHUNKS: *value = s->scratch[0].pool_chunks; return RTGS_OK;
        case RTGS_OPT_KERNEL_TIMING: *value = (int64_t)s->timing_ran.size(); return RTGS_OK;
        case RTGS_OPT_STRIPE: *value = ((int64_t)s->opt_stripe_mod << 32) | (int64_t)s->opt_stripe_rem; return RTGS_OK;
        case RTGS_OPT_MORTON_BITS: *value = s->built ? s->morton_bits_used : s->opt_morton_bits; return RTGS_OK;
        case RTGS_OPT_HEAVY_LISTS: *value = rtgs_heavy_lists_mode(s); return RTGS_OK;
        case RTGS_OPT_HEAVY_LIMIT: *value = s->opt_heavy_limit; return RTGS_OK;
        case RTGS_OPT_TREE_DEPTH:
            if (!s->built) {
                rtgs_set_error("rtgs_scene_get_option(RTGS_OPT_TREE_DEPTH): call rtgs_scene_build_bvh first");
                return RTGS_ERR_STATE;
            }
            *value = s->max_depth;
            return RTGS_OK;
        default:
            rtgs_set_error("unknown option %d", (int)option);
            return RTGS_ERR_INVALID;
    }
}

int rtgs_scene_set_frame_sync(rtgs_scene* s, uint32_t* arrive, const uint32_t* grant, uint32_t grant_value) {
    RTGS_CHECK_ARG(s != nullptr);
    s->sync_arrive = arrive;
    s->sync_grant = grant;
    s->sync_grant_value = grant_value;
    return RTGS_OK;
}

int rtgs_stream_wait_counter(int device, const uint32_t* counter, uint32_t value, void* stream) {
    RTGS_CHECK_ARG(counter != nullptr);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    return rtgs_launch_wait_counter(counter, value, (cudaStream_t)stream);
}

int rtgs_stream_set_counter(int device, uint32_t* counter, uint32_t value, void* stream) {
    RTGS_CHECK_ARG(counter != nullptr);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    return rtgs_launch_set_counter(counter, value, (cudaStream_t)stream);
}

int rtgs_host_register(void* p, size_t bytes) {
    RTGS_CHECK_ARG(p != nullptr && bytes > 0);
    CUDA_TRY(cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return RTGS_OK;
}

int rtgs_host_unregister(void* p) {
    if (p) CUDA_TRY(cudaHostUnregister(p));
    return RTGS_OK;
}

int rtgs_host_device_pointer(void* host, void** dev) {
    RTGS_CHECK_ARG(host != nullptr && dev != nullptr);
    *dev = nullptr;
    CUDA_TRY(cudaHostGetDevicePointer(dev, host, 0));
    return RTGS_OK;
}

int rtgs_stream_store_u32(int device, uint32_t* counter, uint32_t value, void* stream) {
    RTGS_CHECK_ARG(counter != nullptr);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    return rtgs_launch_store_u32(counter, value, (cudaStream_t)stream);
}

static int copy_stripes(int device, float* dst_rgb, const float* dev_rgb, int32_t W, int32_t H, int32_t world,
                        int32_t rank, void* stream, cudaMemcpyKind kind);

int rtgs_copy_stripes_d2h(int device, float* host_rgb, const float* dev_rgb, int32_t W, int32_t H, int32_t world,
                          int32_t rank, void* stream) {
    return copy_stripes(device, host_rgb, dev_rgb, W, H, world, rank, stream, cudaMemcpyDeviceToHost);
}

int rtgs_copy_stripes_d2d(int device, float* dst_rgb, const float* dev_rgb, int32_t W, int32_t H, int32_t world,
                          int32_t rank, void* stream) {
    return copy_stripes(device, dst_rgb, dev_rgb, W, H, world, rank, stream, cudaMemcpyDefault);
}

int rtgs_stream_add_counter(int device, uint32_t* counter, void* stream) {
    RTGS_CHECK_ARG(counter != nullptr);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    return rtgs_launch_add_counter(counter, (cudaStream_t)stream);
}

static int copy_stripes(int device, float* host_rgb, const float* dev_rgb, int32_t W, int32_t H, int32_t world,
                        int32_t rank, void* stream, cudaMemcpyKind kind) {
    RTGS_CHECK_ARG(host_rgb != nullptr && dev_rgb != nullptr);
    RTGS_CHECK_ARG(W > 0 && H > 0 && world >= 1 && rank >= 0 && rank < world);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    // stripe k = pixel columns [32 k, 32 k + 32): 32 * H * 3 contiguous floats of the i-major image; rank owns
    // k = rank, rank + world, ...  All full stripes of the rank move as ONE strided copy (rows = stripes).
    const size_t stripe = (size_t)32 * H * 3 * sizeof(float);
    const int nstripes = (W + 31) / 32;
    const int full = W / 32;                                  // stripes of full width
    const int mine_full = rank < full ? (full - rank + world - 1) / world : 0;
    cudaStream_t st = (cudaStream_t)stream;
    const char* src = reinterpret_cast<const char*>(dev_rgb) + (size_t)rank * stripe;
    char* dst = reinterpret_cast<char*>(host_rgb) + (size_t)rank * stripe;
    if (mine_full > 0)
        CUDA_TRY(cudaMemcpy2DAsync(dst, stripe * world, src, stripe * world, stripe, (size_t)mine_full, kind, st));
    if (nstripes > full && (nstripes - 1) % world == rank) {   // the ragged last stripe
        const size_t off = (size_t)(nstripes - 1) * stripe;
        const size_t bytes = (size_t)(W - 32 * full) * H * 3 * sizeof(float);
        CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(host_rgb) + off, reinterpret_cast<const char*>(dev_rgb) + off,
                                 bytes, kind, st));
    }
    return RTGS_OK;
}

int rtgs_scene_read_kernel_times(rtgs_scene* s, int32_t frames, float* ms) {
    RTGS_CHECK_ARG(s != nullptr && ms != nullptr && frames >= 1);
    const int64_t ring = (int64_t)s->timing_ran.size();
    if (ring == 0 || frames > ring || frames > s->timing_frames) {
        rtgs_set_error("rtgs_scene_read_kernel_times: %d frames requested, %lld timed (ring %lld)", (int)frames,
                       (long long)s->timing_frames, (long long)ring);
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    CUDA_TRY(cudaDeviceSynchronize());
    for (int32_t f = 0; f < frames; ++f) {
        const int64_t slot = (s->timing_frames - frames + f) % ring;
        for (int k = 0; k < RTGS_NUM_KERNELS; ++k) {
            float t = 0.0f;
            if (s->timing_ran[slot] & (1u << k))
                CUDA_TRY(cudaEventElapsedTime(&t, s->timing_events[slot * 4 + k], s->timing_events[slot * 4 + k + 1]));
            ms[f * RTGS_NUM_KERNELS + k] = t;
        }
    }
    return RTGS_OK;
}

int rtgs_host_alloc(size_t bytes, void** out) {
    RTGS_CHECK_ARG(out != nullptr && bytes > 0);
    *out = nullptr;
    CUDA_TRY(cudaHostAlloc(out, bytes, cudaHostAllocPortable | cudaHostAllocMapped));
    return RTGS_OK;
}

int rtgs_host_free(void* p) {
    if (p) CUDA_TRY(cudaFreeHost(p));
    return RTGS_OK;
}

static void* pinned_device_ptr(const void* host) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type != cudaMemoryTypeHost) return nullptr;
    return at.devicePointer;
}

static int check_host_render_args(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                                  int32_t depth, float t_cut, const float* host_rgb, const char* who) {
    RTGS_CHECK_ARG(s != nullptr);
    TRY(check_camera(cam));
    RTGS_CHECK_ARG(host_rgb != nullptr);
    RTGS_CHECK_ARG(w > 0 && h > 0 && x0 >= 0 && y0 >= 0 && x0 + w <= cam->width && y0 + h <= cam->height);
    RTGS_CHECK_ARG(depth >= 1 && depth <= RTGS_MAX_DEPTH);
    RTGS_CHECK_ARG(t_cut >= 0.0f && t_cut < 1.0f);
    if (!s->built) {
        rtgs_set_error("%s: call rtgs_scene_build_bvh first", who);
        return RTGS_ERR_STATE;
    }
    return RTGS_OK;
}

// Banded delivery, first half: launch the frame into a staging slot with the band flags armed.  Region columns
// are contiguous in the (w,h,3) i-major buffer, so a band of macro-tile columns is one contiguous block.
static int submit_banded(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                         int32_t depth, float t_cut, float* host_rgb, float* host_T) {
    rtgs_scene::HostSlot& hs = s->host_slot[s->host_head];
    TRY(ensure_stage(hs, (size_t)w * h));
    const int mrows = (w + 31) / 32;                       // 32-pixel macro-tile columns of the region
    const int bmc = (mrows + 23) / 24 > 0 ? (mrows + 23) / 24 : 1;
    const int nb = (mrows + bmc - 1) / bmc;                // <= 24 bands (RTGS_MAX_BANDS 32)
    for (int b = 0; b < nb; ++b) hs.flags[b] = 0;
    s->bands_active = nb;
    s->band_macro_cols = bmc;
    s->band_flags_cur_dev = hs.flags_dev;
    const int r = rtgs_launch_render(s, cam, x0, y0, w, h, depth, t_cut, 0, 0, hs.stage_rgb,
                                     host_T ? hs.stage_T : nullptr, nullptr, s->own_stream, false);
    s->bands_active = 0;
    s->band_flags_cur_dev = nullptr;
    if (r != RTGS_OK) return r;
    CUDA_TRY(cudaEventRecord(hs.done, s->own_stream));
    hs.nb = nb; hs.bmc = bmc; hs.w = w; hs.h = h;
    hs.host_rgb = host_rgb; hs.host_T = host_T;
    s->host_head ^= 1;
    ++s->host_inflight;
    return RTGS_OK;
}

// Banded delivery, second half, for the oldest frame in flight: the kernels raise a host-visible flag per
// finished band and this thread queues that band's DMA while the later bands (and the next frame, if one has
// been submitted) are still rendering.
static int collect_banded(rtgs_scene* s) {
    rtgs_scene::HostSlot& hs = s->host_slot[s->host_inflight == 2 ? s->host_head : s->host_head ^ 1];
    --s->host_inflight;
    const int nb = hs.nb, bmc = hs.bmc, w = hs.w, h = hs.h, mrows = (w + 31) / 32;
    volatile int* flags = hs.flags;
    int qi = 0;
    for (int b = 0; b < nb; ++b) {
        long spins = 0;
        while (flags[b] == 0) {
            if ((++spins & 0xfff) == 0 && cudaEventQuery(hs.done) != cudaErrorNotReady) break;   // done or failed
        }
        // the band's schedule positions -> macro-tile columns (rotated, render_common.cuh): at most two contiguous
        // runs of columns
        const int p0 = b * bmc, p1 = (b + 1) * bmc < mrows ? (b + 1) * bmc : mrows;
        int lo[2] = {mrows, mrows}, hi[2] = {-1, -1};      // two runs: columns left / right of the middle
        for (int p = p0; p < p1; ++p) {
            const int col = rtgs_dev::macro_column(mrows, p, 2), k = col * 2 >= mrows ? 1 : 0;
            lo[k] = col < lo[k] ? col : lo[k];
            hi[k] = col > hi[k] ? col : hi[k];
        }
        for (int k = 0; k < 2; ++k) {
            if (hi[k] < 0) continue;
            const size_t c0 = (size_t)lo[k] * 32, c1 = (size_t)(hi[k] + 1) * 32 < (size_t)w ? (size_t)(hi[k] + 1) * 32 : (size_t)w;
            cudaStream_t cs = (qi++ & 1) ? s->copy_stream2 : s->copy_stream;
            CUDA_TRY(cudaMemcpyAsync(hs.host_rgb + c0 * h * 3, hs.stage_rgb + c0 * h * 3,
                                     (c1 - c0) * h * 3 * sizeof(float), cudaMemcpyDeviceToHost, cs));
            if (hs.host_T)
                CUDA_TRY(cudaMemcpyAsync(hs.host_T + c0 * h, hs.stage_T + c0 * h, (c1 - c0) * h * sizeof(float),
                                         cudaMemcpyDeviceToHost, cs));
        }
    }
    CUDA_TRY(cudaEventSynchronize(hs.done));
    CUDA_TRY(cudaStreamSynchronize(s->copy_stream));
    CUDA_TRY(cudaStreamSynchronize(s->copy_stream2));
    return RTGS_OK;
}

// Pipelined delivery (rtgs_render_host_submit / _collect).  With a second frame queued behind it, a frame's copy
// does not have to start before the frame is finished: the render runs without band signalling (the per-tile
// release + count costs k_shade_tiles 8 %) and ONE DMA of the whole image follows it on the copy stream, under
// the next frame's render.  No host polling: _collect waits for the copy's event.
static int submit_whole(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                        int32_t depth, float t_cut, float* host_rgb, float* host_T) {
    rtgs_scene::HostSlot& hs = s->host_slot[s->host_head];
    const size_t px = (size_t)w * h;
    TRY(ensure_stage(hs, px));
    // the two frames in flight render on alternating streams (each with its own frame scratch, render.cu), so the
    // head of frame f+1 overlaps the tail of frame f on the device
    cudaStream_t rs = s->host_head == 0 ? s->own_stream : s->own_stream2;
    TRY(rtgs_launch_render(s, cam, x0, y0, w, h, depth, t_cut, 0, 0, hs.stage_rgb, host_T ? hs.stage_T : nullptr, nullptr,
                           rs, false));
    CUDA_TRY(cudaEventRecord(hs.done, rs));
    CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, hs.done, 0));
    CUDA_TRY(cudaMemcpyAsync(host_rgb, hs.stage_rgb, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, s->copy_stream));
    if (host_T)
        CUDA_TRY(cudaMemcpyAsync(host_T, hs.stage_T, px * sizeof(float), cudaMemcpyDeviceToHost, s->copy_stream));
    CUDA_TRY(cudaEventRecord(hs.copied, s->copy_stream));
    hs.nb = 0;   // marks a whole-frame slot for _collect
    s->host_head ^= 1;
    ++s->host_inflight;
    return RTGS_OK;
}

int rtgs_render_host_submit(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                            int32_t depth, float t_cut, float* host_rgb, float* host_T) {
    TRY(check_host_render_args(s, cam, x0, y0, w, h, depth, t_cut, host_rgb, "rtgs_render_host_submit"));
    if (s->host_inflight >= 2) {
        rtgs_set_error("rtgs_render_host_submit: two frames are in flight already; call rtgs_render_host_collect");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    if (!pinned_device_ptr(host_rgb) || (host_T && !pinned_device_ptr(host_T))) {
        rtgs_set_error("rtgs_render_host_submit: the destination must be pinned host memory (rtgs_host_alloc)");
        return RTGS_ERR_INVALID;
    }
    return submit_whole(s, cam, x0, y0, w, h, depth, t_cut, host_rgb, host_T);
}

int rtgs_render_host_submit_packed(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                                   int32_t depth, float t_cut, void* host_pixels, int32_t format) {
    if (format == RTGS_PIXELS_F32)
        return rtgs_render_host_submit(s, cam, x0, y0, w, h, depth, t_cut, (float*)host_pixels, nullptr);
    RTGS_CHECK_ARG(format == RTGS_PIXELS_F16 || format == RTGS_PIXELS_RGBA8);
    TRY(check_host_render_args(s, cam, x0, y0, w, h, depth, t_cut, (const float*)host_pixels,
                               "rtgs_render_host_submit_packed"));
    if (s->host_inflight >= 2) {
        rtgs_set_error("rtgs_render_host_submit_packed: two frames are in flight already; call rtgs_render_host_collect");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    if (!pinned_device_ptr(host_pixels)) {
        rtgs_set_error("rtgs_render_host_submit_packed: the destination must be pinned host memory (rtgs_host_alloc)");
        return RTGS_ERR_INVALID;
    }
    rtgs_scene::HostSlot& hs = s->host_slot[s->host_head];
    const size_t px = (size_t)w * h;
    TRY(ensure_stage(hs, px));
    if (hs.stage_packed_pixels < px) {
        cudaFree(hs.stage_packed);
        hs.stage_packed = nullptr;
        hs.stage_packed_pixels = 0;
        CUDA_TRY(cudaMalloc(&hs.stage_packed, px * 8));
        hs.stage_packed_pixels = px;
    }
    cudaStream_t rs = s->host_head == 0 ? s->own_stream : s->own_stream2;
    TRY(rtgs_launch_render(s, cam, x0, y0, w, h, depth, t_cut, 0, 0, hs.stage_rgb, nullptr, nullptr, rs, false));
    TRY(rtgs_launch_pack_pixels(hs.stage_rgb, hs.stage_packed, (int64_t)px, format, rs));
    CUDA_TRY(cudaEventRecord(hs.done, rs));
    CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, hs.done, 0));
    const size_t bytes = px * (format == RTGS_PIXELS_F16 ? 6 : 4);
    CUDA_TRY(cudaMemcpyAsync(host_pixels, hs.stage_packed, bytes, cudaMemcpyDeviceToHost, s->copy_stream));
    CUDA_TRY(cudaEventRecord(hs.copied, s->copy_stream));
    hs.nb = 0;   // a whole-frame slot for _collect
    s->host_head ^= 1;
    ++s->host_inflight;
    return RTGS_OK;
}

int rtgs_render_host_collect(rtgs_scene* s) {
    RTGS_CHECK_ARG(s != nullptr);
    if (s->host_inflight <= 0) {
        rtgs_set_error("rtgs_render_host_collect: no frame in flight");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    rtgs_scene::HostSlot& hs = s->host_slot[s->host_inflight == 2 ? s->host_head : s->host_head ^ 1];
    if (hs.nb > 0) return collect_banded(s);
    --s->host_inflight;
    CUDA_TRY(cudaEventSynchronize(hs.copied));
    return RTGS_OK;
}

int rtgs_render_host(rtgs_scene* s, const rtgs_camera* cam, int32_t x0, int32_t y0, int32_t w, int32_t h,
                     int32_t depth, float t_cut, float* host_rgb, float* host_T) {
    TRY(check_host_render_args(s, cam, x0, y0, w, h, depth, t_cut, host_rgb, "rtgs_render_host"));
    if (s->host_inflight != 0) {
        rtgs_set_error("rtgs_render_host: %d submitted frame(s) not collected yet", s->host_inflight);
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    if (pinned_device_ptr(host_rgb) && (!host_T || pinned_device_ptr(host_T))) {
        // a pinned destination: the band copies run while the later bands are still rendering
        TRY(submit_banded(s, cam, x0, y0, w, h, depth, t_cut, host_rgb, host_T));
        return collect_banded(s);
    }
    // pageable memory: render, one DMA into the scene's pinned buffer, then a host copy
    const size_t px = (size_t)w * h;
    cudaStream_t st = s->own_stream;
    rtgs_scene::HostSlot& hs = s->host_slot[0];
    TRY(ensure_stage(hs, px));
    TRY(rtgs_launch_render(s, cam, x0, y0, w, h, depth, t_cut, 0, 0, hs.stage_rgb, host_T ? hs.stage_T : nullptr, nullptr,
                           st, false));
    TRY(ensure_pinned(s, px));
    CUDA_TRY(cudaMemcpyAsync(s->pinned_rgb, hs.stage_rgb, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (host_T) CUDA_TRY(cudaMemcpyAsync(s->pinned_T, hs.stage_T, px * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    memcpy(host_rgb, s->pinned_rgb, px * 3 * sizeof(float));
    if (host_T) memcpy(host_T, s->pinned_T, px * sizeof(float));
    return RTGS_OK;
}

int rtgs_device_alloc(int device, size_t bytes, void** out) {
    RTGS_CHECK_ARG(out != nullptr && bytes > 0);
    *out = nullptr;
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    CUDA_TRY(cudaMalloc(out, bytes));
    return RTGS_OK;
}

int rtgs_device_free(int device, void* p) {
    DeviceGuard g(device);
    if (p) CUDA_TRY(cudaFree(p));
    return RTGS_OK;
}

int rtgs_ipc_export(int device, const void* dev_ptr, unsigned char* handle) {
    RTGS_CHECK_ARG(dev_ptr != nullptr && handle != nullptr);
    static_assert(sizeof(cudaIpcMemHandle_t) == RTGS_IPC_HANDLE_BYTES, "handle size");
    DeviceGuard g(device);
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, const_cast<void*>(dev_ptr)));
    memcpy(handle, &h, sizeof(h));
    return RTGS_OK;
}

int rtgs_ipc_open(int device, const unsigned char* handle, void** out) {
    RTGS_CHECK_ARG(handle != nullptr && out != nullptr);
    *out = nullptr;
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CUDA_TRY(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return RTGS_OK;
}

int rtgs_ipc_close(int device, void* p) {
    DeviceGuard g(device);
    if (p) CUDA_TRY(cudaIpcCloseMemHandle(p));
    return RTGS_OK;
}

int rtgs_generate_rays(const rtgs_camera* cam, int device, float* rays, void* stream) {
    TRY(check_camera(cam));
    RTGS_CHECK_ARG(rays != nullptr);
    DeviceGuard g(device);
    if (!g.ok) {
        rtgs_set_error("cudaSetDevice(%d) failed", device);
        return RTGS_ERR_CUDA;
    }
    return rtgs_launch_generate_rays(cam, rays, (cudaStream_t)stream);
}

int rtgs_trace_closest(rtgs_scene* s, int64_t nrays, const float* rays, int32_t* idx, float* t12, void* stream) {
    RTGS_CHECK_ARG(s != nullptr);
    RTGS_CHECK_ARG(nrays >= 0);
    RTGS_CHECK_ARG(nrays == 0 || (rays && idx && t12));
    if (!s->built) {
        rtgs_set_error("rtgs_trace_closest: call rtgs_scene_build_bvh first");
        return RTGS_ERR_STATE;
    }
    DeviceGuard g(s->device);
    return rtgs_launch_trace_closest(s, nrays, rays, idx, t12, (cudaStream_t)stream);
}

int rtgs_render_rays(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut, float* out_rgb,
                     float* out_T, void* stream) {
    return rtgs_render_rays_depth(s, nrays, rays, depth, t_cut, out_rgb, out_T, nullptr, stream);
}

int rtgs_render_rays_depth(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                           float* out_rgb, float* out_T, float* out_depth, void* stream) {
    TRY(check_rays(s, nrays, rays, out_rgb, depth, t_cut));
    RTGS_CHECK_ARG(aligned(out_T, 4) && aligned(out_depth, 4));
    if (!s->built) {
        rtgs_set_error("%s: call rtgs_scene_build_bvh first", out_depth ? "rtgs_render_rays_depth" : "rtgs_render_rays");
        return RTGS_ERR_STATE;
    }
    if (nrays == 0) return RTGS_OK;
    DeviceGuard g(s->device);
    return rtgs_launch_render_rays(s, nrays, rays, depth, t_cut, out_rgb, out_T, out_depth, (cudaStream_t)stream);
}

int rtgs_render_rays_backward(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                              const float* dL_drgb, const float* dL_dT, float* grad_pos, float* grad_rot,
                              float* grad_scale, float* grad_color, float* grad_opacity, float* grad_sh,
                              float* grad_rays, float* replay_rgb, float* replay_T, void* stream) {
    return rtgs_render_rays_backward_depth(s, nrays, rays, depth, t_cut, dL_drgb, dL_dT, grad_pos, grad_rot,
                                           grad_scale, grad_color, grad_opacity, grad_sh, grad_rays, replay_rgb,
                                           replay_T, nullptr, nullptr, stream);
}

int rtgs_render_rays_backward_depth(rtgs_scene* s, int64_t nrays, const float* rays, int32_t depth, float t_cut,
                                    const float* dL_drgb, const float* dL_dT, float* grad_pos, float* grad_rot,
                                    float* grad_scale, float* grad_color, float* grad_opacity, float* grad_sh,
                                    float* grad_rays, float* replay_rgb, float* replay_T, const float* dL_dD,
                                    float* replay_depth, void* stream) {
    TRY(check_rays(s, nrays, rays, dL_drgb, depth, t_cut));
    float* const grads[6] = {grad_pos, grad_rot, grad_scale, grad_color, grad_opacity, grad_sh};
    for (const float* p : grads) RTGS_CHECK_ARG(aligned(p, 4));
    RTGS_CHECK_ARG(aligned(dL_dT, 4) && aligned(grad_rays, 4) && aligned(replay_rgb, 4) && aligned(replay_T, 4));
    RTGS_CHECK_ARG(aligned(dL_dD, 4) && aligned(replay_depth, 4));
    const bool with_depth = dL_dD != nullptr || replay_depth != nullptr;
    if (!s->built) {
        rtgs_set_error("%s: call rtgs_scene_build_bvh first",
                       with_depth ? "rtgs_render_rays_backward_depth" : "rtgs_render_rays_backward");
        return RTGS_ERR_STATE;
    }
    if (nrays == 0) return RTGS_OK;
    DeviceGuard g(s->device);
    return rtgs_launch_render_rays_backward(s, nrays, rays, depth, t_cut, dL_drgb, dL_dT, dL_dD, grads, grad_rays,
                                            replay_rgb, replay_T, replay_depth, (cudaStream_t)stream);
}

int rtgs_scene_destroy(rtgs_scene* s) {
    free_scene(s);
    return RTGS_OK;
}

}  // extern "C"
