"""ctypes binding of the C-ABI in include/rtgs_b200.h (librtgs_b200.so).

There is NO CPU fallback: if the CUDA library is missing or fails to load, importing the render
path raises.  Build it with ``python rt-gaussian-splat-renderer_b200/build.py``.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent.parent
LIB_PATH = Path(os.environ.get("RTGS_B200_LIB", _PKG / "lib" / "librtgs_b200.so"))


class RtgsError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"rtgs_b200 error {status}: {message}")
        self.status = status


class rtgs_camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("rotation", C.c_float * 4), ("focal", C.c_float * 2),
                ("width", C.c_int32), ("height", C.c_int32)]


class rtgs_render_stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays", "rays_hit", "layers", "nodes_tested", "candidates",
                                          "pair_tests", "f64_refinements", "tiles", "traversal_steps",
                                          "insert_rounds", "fallback_tiles", "useful_candidates",
                                          "max_lists_stack", "max_fused_stack", "max_group_list",
                                          "heavy_groups", "heavy_failed", "heavy_passes", "heavy_sample_tests",
                                          "max_deferred", "heavy_retries", "heavy_failed_list",
                                          "heavy_failed_deferred", "heavy_failed_passes",
                                          "heavy_cycles_walk", "heavy_cycles_test", "heavy_cycles_publish")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


_fp = C.POINTER(C.c_float)
_vp = C.c_void_p

#: every symbol include/rtgs_b200.h declares -> (restype, argtypes)
SIGNATURES = {
    "rtgs_last_error": (C.c_char_p, []),
    "rtgs_abi_version": (C.c_int, []),
    "rtgs_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "rtgs_scene_create": (C.c_int, [C.c_int, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "rtgs_scene_create_from_ply_rows": (C.c_int, [C.c_int, C.c_int64, _vp, C.c_int32, _vp, C.c_float,
                                                  C.c_int32, C.POINTER(_vp)]),
    "rtgs_scene_build_bvh": (C.c_int, [_vp, C.c_int32]),
    "rtgs_scene_build_ms": (C.c_int, [_vp, C.POINTER(C.c_float)]),
    "rtgs_scene_morton_bits": (C.c_int, [_vp, C.POINTER(C.c_int32)]),
    "rtgs_scene_num_gaussians": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "rtgs_scene_device": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "rtgs_scene_read_lbvh": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_scene_read_morton64": (C.c_int, [_vp, _vp]),
    "rtgs_scene_read_gaussians": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_render": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                              C.c_int32, C.c_float, C.c_int32, C.c_int32, _vp, _vp, _vp,
                              C.POINTER(rtgs_render_stats)]),
    "rtgs_render_depth": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_float, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp,
                                    C.POINTER(rtgs_render_stats)]),
    "rtgs_scene_set_gaussians_device": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_render_backward": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_int32, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _vp]),
    "rtgs_render_backward_camera": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32,
                                              C.c_int32, C.c_int32, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                              _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_render_backward_depth": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32,
                                             C.c_int32, C.c_int32, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                             _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_scene_set_option": (C.c_int, [_vp, C.c_int32, C.c_int64]),
    "rtgs_scene_get_option": (C.c_int, [_vp, C.c_int32, C.POINTER(C.c_int64)]),
    "rtgs_scene_set_frame_sync": (C.c_int, [_vp, _vp, _vp, C.c_uint32]),
    "rtgs_stream_wait_counter": (C.c_int, [C.c_int, _vp, C.c_uint32, _vp]),
    "rtgs_stream_set_counter": (C.c_int, [C.c_int, _vp, C.c_uint32, _vp]),
    "rtgs_host_register": (C.c_int, [_vp, C.c_size_t]),
    "rtgs_host_unregister": (C.c_int, [_vp]),
    "rtgs_host_device_pointer": (C.c_int, [_vp, C.POINTER(_vp)]),
    "rtgs_stream_store_u32": (C.c_int, [C.c_int, _vp, C.c_uint32, _vp]),
    "rtgs_copy_stripes_d2h": (C.c_int, [C.c_int, _vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp]),
    "rtgs_copy_stripes_d2d": (C.c_int, [C.c_int, _vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp]),
    "rtgs_stream_add_counter": (C.c_int, [C.c_int, _vp, _vp]),
    "rtgs_scene_read_kernel_times": (C.c_int, [_vp, C.c_int32, _vp]),
    "rtgs_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp)]),
    "rtgs_host_free": (C.c_int, [_vp]),
    "rtgs_device_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(_vp)]),
    "rtgs_device_free": (C.c_int, [C.c_int, _vp]),
    "rtgs_ipc_export": (C.c_int, [C.c_int, _vp, _vp]),
    "rtgs_ipc_open": (C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    "rtgs_ipc_close": (C.c_int, [C.c_int, _vp]),
    "rtgs_render_host": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_float, _vp, _vp]),
    "rtgs_render_host_submit": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_float, _vp, _vp]),
    "rtgs_render_host_collect": (C.c_int, [_vp]),
    "rtgs_render_host_submit_packed": (C.c_int, [_vp, C.POINTER(rtgs_camera), C.c_int32, C.c_int32, C.c_int32,
                                                 C.c_int32, C.c_int32, C.c_float, _vp, C.c_int32]),
    "rtgs_generate_rays": (C.c_int, [C.POINTER(rtgs_camera), C.c_int, _vp, _vp]),
    "rtgs_trace_closest": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp]),
    "rtgs_render_rays": (C.c_int, [_vp, C.c_int64, _vp, C.c_int32, C.c_float, _vp, _vp, _vp]),
    "rtgs_render_rays_depth": (C.c_int, [_vp, C.c_int64, _vp, C.c_int32, C.c_float, _vp, _vp, _vp, _vp]),
    "rtgs_render_rays_backward": (C.c_int, [_vp, C.c_int64, _vp, C.c_int32, C.c_float, _vp, _vp, _vp, _vp, _vp,
                                            _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_render_rays_backward_depth": (C.c_int, [_vp, C.c_int64, _vp, C.c_int32, C.c_float, _vp, _vp, _vp, _vp,
                                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rtgs_scene_destroy": (C.c_int, [_vp]),
}

OPT_RENDER_MODE, OPT_LIST_POOL_CHUNKS, OPT_KERNEL_TIMING, OPT_STRIPE, OPT_MORTON_BITS, OPT_TREE_DEPTH = 0, 1, 2, 3, 4, 5
OPT_HEAVY_LISTS, OPT_HEAVY_LIMIT = 6, 7
#: the (up to) three launches of a frame, by render mode (rtgs_scene_read_kernel_times); None = no launch
KERNEL_NAMES_BY_MODE = {0: ("k_tile_lists", "k_shade_tiles", "k_render"),
                        1: (None, None, "k_render"),
                        2: (None, "k_frame", "k_render")}
KERNEL_NAMES = KERNEL_NAMES_BY_MODE[0]
#: rtgs_pixel_format: name -> (enum value, numpy dtype, channels)
PIXEL_FORMATS = {"f32": (0, "float32", 3), "f16": (1, "float16", 3), "rgba8": (2, "uint8", 4)}

_lib = None


def load():
    """Load the shared library (once) and bind every declared symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} not found: the rtgs render path is CUDA-only (no CPU fallback). "
            f"Build it with `python {(_PKG / 'build.py')}`.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        msg = load().rtgs_last_error()
        raise RtgsError(status, msg.decode() if msg else "")


def make_camera(position, rotation, focal, width, height) -> rtgs_camera:
    cam = rtgs_camera()
    cam.position[:] = [float(v) for v in position]
    cam.rotation[:] = [float(v) for v in rotation]
    cam.focal[:] = [float(v) for v in focal]
    cam.width, cam.height = int(width), int(height)
    return cam


def device_count() -> int:
    n = C.c_int(0)
    check(load().rtgs_device_count(C.byref(n)))
    return n.value


class PinnedBuffer:
    """A pinned, device-mapped host buffer (rtgs_host_alloc).  ``view()`` returns a NumPy array over it;
    every view keeps the buffer alive, so the memory is released only after the last view is gone."""

    def __init__(self, shape, dtype="float32"):
        import numpy as np
        self.shape = tuple(int(v) for v in shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(load().rtgs_host_alloc(self.nbytes, C.byref(p)))
        self._ptr = p

    @property
    def ptr(self):
        return self._ptr.value

    def view(self):
        import numpy as np
        buf = (C.c_char * self.nbytes).from_address(self._ptr.value)
        buf._owner = self          # the ndarray's base keeps `buf`, which keeps this buffer alive
        return np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def __del__(self):
        try:
            if self._ptr is not None and self._ptr.value:
                load().rtgs_host_free(self._ptr)
                self._ptr = None
        except Exception:
            pass
