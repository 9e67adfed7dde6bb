"""Gaussian-splatting scene — B200-native mirror of the reference's ``rtgs/scene.py``.

Keeps the reference's surface (``Scene(max_num_node, balance_weight, leaf_prim)``,
``load_file(path, scale)``, ``gaussian_field``, ``bvh_field``, ``hit``; scene.py:64-450) on top of
the C-ABI: the Gaussians live in packed device records, and the reference's host-driven binned-SAH
builder (scene.py:162-404) is replaced by a GPU LBVH (csrc/lbvh.cu).  There is no CPU fallback.
"""
from __future__ import annotations

import collections
import ctypes as C
import logging
import pathlib
from dataclasses import dataclass

import numpy as np

from . import _native
from .bvh import BVH_DTYPE, BVHNode
from .fields import StructArrayField
from .gaussian import GAUSSIAN_DTYPE, SH_NAMES, Gaussian
from .ply import read_ply
from .ray import RAY_DTYPE
from .utils.math import sigmoid

logger = logging.getLogger(__name__)


@dataclass
class SceneHit:
    """Scene hit information (scene.py:24-33), batched: one entry per ray.

    gaussian_idx: index into ``Scene.gaussian_field`` (-1 = miss); intersections: (t1, t2);
    depth: depth of the LBVH leaf holding the Gaussian (-1 on a miss)."""
    gaussian_idx: np.ndarray
    intersections: np.ndarray
    depth: np.ndarray


def _f32(a, shape):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.shape != shape:
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a


def _default_device() -> int:
    try:
        import torch
        if torch.cuda.is_available():
            return int(torch.cuda.current_device())
    except ImportError:
        pass
    return 0


class Scene:
    """A Gaussian splatting scene (scene.py:64-87).

    max_num_node and balance_weight configured the reference's SAH builder; the LBVH always has
    2n-1 nodes and no balance heuristic, so both are accepted and ignored.  leaf_prim is passed to
    the builder (LBVH leaves currently hold one Gaussian)."""

    def __init__(self, max_num_node: int = 128, balance_weight: int = 1, leaf_prim=8, device: int | None = None,
                 morton_bits: int | str = "auto"):
        self.max_num_node = max_num_node
        self.balance_weight = balance_weight
        self.leaf_prim = leaf_prim
        self.device = device
        if morton_bits not in ("auto", 0, 30, 63):
            raise ValueError('morton_bits must be "auto", 30 or 63')
        # LBVH code width requested: "auto" = 30 bits unless they do not resolve the scene (far outliers), then 63;
        # after the build `morton_bits` is the width in use.  The image does not depend on it.
        self._morton_request = 0 if morton_bits in ("auto", 0) else int(morton_bits)
        self.morton_bits = 30
        self._handle = None
        self._n = 0
        self._gaussian_field = None
        self._bvh_field = None
        self._lbvh = None
        self.has_sh = False
        self._pending = collections.deque()   # frames queued by RayTracer.render_async, oldest first

    # ------------------------------------------------------------------ construction
    def load_file(self, path: pathlib.Path, scale: float = 1, sh_layout: str = "channel_major",
                  activate_on_device: bool = False):
        """Load a 3DGS ``.ply`` (scene.py:89-160) and build the BVH (scene.py:162-404).

        The activations are the reference's NumPy float32 expressions (scene.py:101-114) unless
        ``activate_on_device`` selects the fused CUDA ingest (rtgs_scene_create_from_ply_rows).
        sh_layout - how the 45 ``f_rest_*`` columns become the 15 RGB triples ``sh_10 .. sh_36``.  The reference
        reshapes them to (N,3,15) and copies that array into an (N,15) field of vec3 without a transpose
        (scene.py:106-107,122,127); what real Taichi 1.7.3 stores then cannot be established offline, so the
        layouts are named for what they DO, not for what Taichi is believed to do:
          "channel_major"  sh_k[c] = f_rest_{15c+k}: the standard 3DGS file layout, the evident intent of
                           ``reshape((-1,3,15))``; the default here;
          "interleaved"    sh_k[c] = f_rest_{3k+c}: the flat C-order reinterpretation of that (N,3,15) buffer as
                           (N,15,3), which is what ``oracle/taichi_shim`` executes and therefore what the committed
                           reference-run goldens contain.  (SURVEY.md §7 hard part 7 derives yet another candidate
                           for real Taichi, flat[45i+15k+c] with out-of-row reads; none of the three is verified.)
        ``"taichi_as_executed"`` is accepted as a deprecated alias of "interleaved".
        """
        path = pathlib.Path(path)
        cols = read_ply(path.resolve())
        num_points = len(cols["x"])
        logger.info(f"Point cloud loaded from {path} with {num_points} points.")
        if sh_layout == "taichi_as_executed":
            sh_layout = "interleaved"
        if sh_layout not in ("channel_major", "interleaved"):
            raise ValueError(sh_layout)
        if activate_on_device:
            return self._load_rows_on_device(cols, scale, sh_layout)
        positions = np.stack([cols["x"], cols["y"], cols["z"]], axis=-1)
        # Convert quaternion order from scalar first to scalar last (scene.py:103).
        rotations = np.stack([cols["rot_1"], cols["rot_2"], cols["rot_3"], cols["rot_0"]], axis=-1)
        scales = np.stack([cols["scale_0"], cols["scale_1"], cols["scale_2"]], axis=-1)
        colors = np.stack([cols["f_dc_0"], cols["f_dc_1"], cols["f_dc_2"]], axis=-1)
        opacities = cols["opacity"]
        rotations = rotations / np.linalg.norm(rotations, axis=-1)[:, np.newaxis]   # scene.py:110-111
        scales = np.exp(scales) * np.float32(scale)                                  # scene.py:112
        colors = sigmoid(colors)                                                     # scene.py:113
        opacities = sigmoid(opacities)                                               # scene.py:114
        sh = None
        if all(f"f_rest_{i}" in cols for i in range(45)):
            rest = np.stack([cols[f"f_rest_{i}"] for i in range(45)], axis=-1)
            if sh_layout == "channel_major":
                sh = rest.reshape(-1, 3, 15).transpose(0, 2, 1)
            else:
                sh = rest.reshape(-1, 15, 3)
        self.from_arrays(positions, rotations, scales, colors, opacities, sh)
        logger.info("Gaussian field loaded successfully.")
        return self

    def _load_rows_on_device(self, cols, scale, sh_layout):
        names = (["x", "y", "z", "f_dc_0", "f_dc_1", "f_dc_2"] + [f"f_rest_{i}" for i in range(45)]
                 + ["opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"])
        present = [n for n in names if n in cols]
        rows = np.ascontiguousarray(np.stack([np.asarray(cols[n], dtype=np.float32) for n in present], axis=-1))
        col = np.array([present.index(n) if n in cols else -1 for n in names], dtype=np.int32)
        lib = _native.load()
        self._release()
        dev = _default_device() if self.device is None else int(self.device)
        h = C.c_void_p()
        _native.check(lib.rtgs_scene_create_from_ply_rows(
            dev, rows.shape[0], rows.ctypes.data, rows.shape[1], col.ctypes.data, float(scale),
            0 if sh_layout == "channel_major" else 1, C.byref(h)))
        self._adopt(h, rows.shape[0], dev, any(f"f_rest_{i}" in cols for i in range(45)))
        return self

    def from_arrays(self, pos, rot_xyzw, scale, color, opacity, sh=None):
        """Build the scene from POST-activation parameter arrays (additive API for synthetic scenes):
        pos (n,3), rot_xyzw (n,4) unit, scale (n,3) linear, color (n,3), opacity (n,), sh (n,15,3)|None."""
        pos = np.ascontiguousarray(pos, dtype=np.float32)
        n = pos.shape[0]
        if n < 1:
            raise ValueError("a scene needs at least one Gaussian")
        pos = _f32(pos, (n, 3))
        rot = _f32(rot_xyzw, (n, 4))
        sca = _f32(scale, (n, 3))
        col = _f32(color, (n, 3))
        opa = _f32(np.asarray(opacity).reshape(n), (n,))
        shp = None if sh is None else _f32(np.asarray(sh).reshape(n, 15, 3), (n, 15, 3))
        lib = _native.load()
        self._release()
        dev = _default_device() if self.device is None else int(self.device)
        h = C.c_void_p()
        _native.check(lib.rtgs_scene_create(dev, n, pos.ctypes.data, rot.ctypes.data, sca.ctypes.data,
                                            col.ctypes.data, opa.ctypes.data,
                                            None if shp is None else shp.ctypes.data, C.byref(h)))
        self._adopt(h, n, dev, shp is not None)
        return self

    def set_gaussians(self, pos, rot, scale, color, opacity, sh=None):
        """Replace the stored parameters in place from CUDA float32 tensors on the scene's device and rebuild the
        LBVH (rtgs_scene_set_gaussians_device + rtgs_scene_build_bvh): no host round trip, same handle.  Shapes as
        in ``from_arrays`` (n fixed); ``sh`` must be given iff the scene has SH.  The copies are ordered after the
        work already queued on the current stream."""
        import torch
        n = self._n
        dev = torch.device("cuda", self.device)
        want = dict(pos=(n, 3), rot=(n, 4), scale=(n, 3), color=(n, 3), opacity=(n,))
        args = dict(pos=pos, rot=rot, scale=scale, color=color, opacity=opacity)
        if (sh is not None) != self.has_sh:
            raise ValueError("sh must be given iff the scene has SH coefficients")
        if sh is not None:
            want["sh"], args["sh"] = (n, 15, 3), sh
        for name, t in args.items():
            if not isinstance(t, torch.Tensor) or t.device != dev or t.dtype != torch.float32:
                raise ValueError(f"{name}: expected a float32 tensor on {dev}")
            if tuple(t.shape) != want[name] or not t.is_contiguous():
                raise ValueError(f"{name}: expected a contiguous tensor of shape {want[name]}, got {tuple(t.shape)}")
        self.drain_pending()
        lib = _native.load()
        stream = torch.cuda.current_stream(dev).cuda_stream
        _native.check(lib.rtgs_scene_set_gaussians_device(
            self.handle, pos.data_ptr(), rot.data_ptr(), scale.data_ptr(), color.data_ptr(), opacity.data_ptr(),
            None if sh is None else sh.data_ptr(), stream))
        self._gaussian_field = self._bvh_field = self._lbvh = None
        _native.check(lib.rtgs_scene_build_bvh(self.handle, int(self.leaf_prim)))
        bits = C.c_int32()
        _native.check(lib.rtgs_scene_morton_bits(self.handle, C.byref(bits)))
        self.morton_bits = int(bits.value)
        return self

    def _adopt(self, handle, n, dev, has_sh):
        self._handle = handle
        self._n = int(n)
        self.device = dev
        self.has_sh = bool(has_sh)
        self._gaussian_field = self._bvh_field = self._lbvh = None
        _native.check(_native.load().rtgs_scene_set_option(self._handle, _native.OPT_MORTON_BITS,
                                                           self._morton_request))
        _native.check(_native.load().rtgs_scene_build_bvh(self._handle, int(self.leaf_prim)))
        bits = C.c_int32()
        _native.check(_native.load().rtgs_scene_morton_bits(self._handle, C.byref(bits)))
        self.morton_bits = int(bits.value)
        logger.info(f"Build {2 * self._n - 1} BVH nodes in total ({self.build_ms:.2f} ms on the device). "
                    "Max leaf node size is 1.")

    def drain_pending(self):
        """Collect every frame queued by ``RayTracer.render_async`` (the synchronous calls do this first)."""
        while self._pending:
            self._pending[0].result()

    def _release(self):
        if self._handle is not None:
            self._pending.clear()
            _native.load().rtgs_scene_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    # ------------------------------------------------------------------ accessors
    @property
    def handle(self):
        if self._handle is None:
            raise RuntimeError("scene is empty: call load_file() or from_arrays() first")
        return self._handle

    @property
    def build_ms(self) -> float:
        """Device time of the LBVH build (ms)."""
        ms = C.c_float()
        _native.check(_native.load().rtgs_scene_build_ms(self.handle, C.byref(ms)))
        return float(ms.value)

    @property
    def num_gaussians(self) -> int:
        return self._n

    _OPTIONS = {"render_mode": _native.OPT_RENDER_MODE, "list_pool_chunks": _native.OPT_LIST_POOL_CHUNKS,
                "kernel_timing": _native.OPT_KERNEL_TIMING, "stripe": _native.OPT_STRIPE,
                "morton_bits": _native.OPT_MORTON_BITS, "tree_depth": _native.OPT_TREE_DEPTH,
                "heavy_lists": _native.OPT_HEAVY_LISTS, "heavy_limit": _native.OPT_HEAVY_LIMIT}

    def set_option(self, name: str, value: int) -> "Scene":
        """Render-path tuning (rtgs_scene_set_option): ``render_mode`` 0 = tile lists + shading kernels (default),
        2 = the whole frame in one launch (k_frame), 1 = the fused kernel alone; ``list_pool_chunks`` = capacity of
        the candidate-list pool (-1 = default)."""
        _native.check(_native.load().rtgs_scene_set_option(self.handle, self._OPTIONS[name], int(value)))
        return self

    def get_option(self, name: str) -> int:
        """Current value of an option (rtgs_scene_get_option); ``tree_depth`` (read-only) is the depth of the
        deepest LBVH leaf."""
        v = C.c_int64()
        _native.check(_native.load().rtgs_scene_get_option(self.handle, self._OPTIONS[name], C.byref(v)))
        return int(v.value)

    @property
    def render_mode(self) -> int:
        return self.get_option("render_mode")

    @property
    def kernel_names(self):
        """Names of the frame's (up to) three launches in the current render mode (None = no launch)."""
        return _native.KERNEL_NAMES_BY_MODE[self.render_mode]

    def set_frame_sync(self, arrive: int = 0, grant: int = 0, grant_value: int = 0) -> "Scene":
        """Multi-GPU hand-over of the NEXT frame (rtgs_scene_set_frame_sync): device addresses of 32-bit counters,
        0 = none.  Used by ``rtgs.sharding.PeerFrame``."""
        _native.check(_native.load().rtgs_scene_set_frame_sync(self.handle, arrive or None, grant or None,
                                                               int(grant_value) & 0xffffffff))
        return self

    def set_stripe(self, world: int = 1, rank: int = 0) -> "Scene":
        """Tile sharding of one frame: following renders touch only the 32-column stripes k with k % world == rank
        (rtgs.sharding.STRIPE_COLUMNS); ``set_stripe()`` restores full frames."""
        return self.set_option("stripe", (int(world) << 32) | int(rank))

    def read_kernel_times(self, frames: int):
        """(frames, 3) float32 milliseconds of the frame's launches (``kernel_names``) for the last `frames` renders
        (needs ``set_option("kernel_timing", n)`` with n >= frames beforehand).  Synchronises the device."""
        out = np.zeros((int(frames), len(_native.KERNEL_NAMES)), np.float32)
        _native.check(_native.load().rtgs_scene_read_kernel_times(self.handle, int(frames), out.ctypes.data))
        return out

    def read_gaussians(self) -> dict:
        """Stored parameters in original order as float32 arrays."""
        n = self._n
        out = dict(pos=np.empty((n, 3), np.float32), rot=np.empty((n, 4), np.float32),
                   scale=np.empty((n, 3), np.float32), color=np.empty((n, 3), np.float32),
                   opacity=np.empty((n,), np.float32), sh=np.empty((n, 15, 3), np.float32))
        _native.check(_native.load().rtgs_scene_read_gaussians(
            self.handle, out["pos"].ctypes.data, out["rot"].ctypes.data, out["scale"].ctypes.data,
            out["color"].ctypes.data, out["opacity"].ctypes.data, out["sh"].ctypes.data))
        if not self.has_sh:
            out["sh"] = None
        return out

    def read_lbvh(self) -> dict:
        """LBVH integers and boxes (parity read-back): morton (n; uint64 for morton_bits=63) in original order, sorted_idx (n),
        child (n-1,2) unified ids (leaf k -> n-1+k), parent (2n-1), aabb (2n-1,6)."""
        if self._lbvh is None:
            n = self._n
            wide = self.morton_bits == 63
            out = dict(morton=np.empty(n, np.uint64 if wide else np.uint32), sorted_idx=np.empty(n, np.uint32),
                       child=np.empty((max(n - 1, 0), 2), np.int32), parent=np.empty(2 * n - 1, np.int32),
                       aabb=np.empty((2 * n - 1, 6), np.float32))
            if wide:
                _native.check(_native.load().rtgs_scene_read_morton64(self.handle, out["morton"].ctypes.data))
            _native.check(_native.load().rtgs_scene_read_lbvh(
                self.handle, None if wide else out["morton"].ctypes.data, out["sorted_idx"].ctypes.data,
                out["child"].ctypes.data if n > 1 else None, out["parent"].ctypes.data, out["aabb"].ctypes.data))
            self._lbvh = out
        return self._lbvh

    @property
    def gaussian_field(self):
        """``Gaussian.field(shape=(n,))`` view of the stored parameters (scene.py:131), original order."""
        if self._handle is None:
            return Gaussian.field(shape=())
        if self._gaussian_field is None:
            g = self.read_gaussians()
            a = np.zeros(self._n, dtype=GAUSSIAN_DTYPE)
            a["position"], a["rotation"], a["scale"] = g["pos"], g["rot"], g["scale"]
            a["color"], a["opacity"] = g["color"], g["opacity"]
            if g["sh"] is not None:
                for k, name in enumerate(SH_NAMES):
                    a[name] = g["sh"][:, k, :]
            self._gaussian_field = StructArrayField(a, Gaussian._from_record)
        return self._gaussian_field

    @property
    def bvh_field(self):
        """The LBVH in the reference's node record shape (bvh.py:10-17): 2n-1 nodes, root 0;
        prim_left/prim_right index the Morton-sorted order (``read_lbvh()['sorted_idx']``)."""
        if self._handle is None:
            return BVHNode.field(shape=(self.max_num_node,))
        if self._bvh_field is None:
            lb = self.read_lbvh()
            n = self._n
            a = np.zeros(2 * n - 1, dtype=BVH_DTYPE)
            a["p_min"], a["p_max"] = lb["aabb"][:, :3], lb["aabb"][:, 3:]
            a["left"] = a["right"] = -1
            if n > 1:
                a["left"][: n - 1] = lb["child"][:, 0]
                a["right"][: n - 1] = lb["child"][:, 1]
            # leaf ranges, then propagate to parents level by level; depth from the root
            first = np.zeros(2 * n - 1, np.int64)
            last = np.zeros(2 * n - 1, np.int64)
            first[n - 1:] = np.arange(n)
            last[n - 1:] = np.arange(n) + 1
            depth = np.zeros(2 * n - 1, np.int32)
            if n > 1:
                child = lb["child"]
                levels = []
                frontier = np.array([0])
                while frontier.size:
                    levels.append(frontier)
                    kids = child[frontier].reshape(-1)
                    depth[kids] = np.repeat(depth[frontier] + 1, 2)
                    frontier = kids[kids < n - 1]
                for nodes in reversed(levels):   # leaf ranges propagate bottom-up, one level at a time
                    l, r = child[nodes, 0], child[nodes, 1]
                    first[nodes] = np.minimum(first[l], first[r])
                    last[nodes] = np.maximum(last[l], last[r])
            a["prim_left"], a["prim_right"], a["depth"] = first, last, depth
            self._bvh_field = StructArrayField(a, BVHNode._from_record)
        return self._bvh_field

    # ------------------------------------------------------------------ Scene.hit
    def hit(self, rays) -> SceneHit:
        """Closest-entry ray cast for a batch of rays (scene.py:406-450).

        rays: a ``Ray``, a structured array of ``RAY_DTYPE`` or an (n,8) float array
        (origin, direction, start, end).  Returns batched ``SceneHit``."""
        import torch
        from .ray import Ray
        if isinstance(rays, Ray):
            rays = rays.to_record().reshape(1)
        rays = np.asarray(rays)
        if rays.dtype == RAY_DTYPE:
            rays = np.ascontiguousarray(rays).view(np.float32).reshape(-1, 8)
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
        n = rays.shape[0]
        dev = torch.device("cuda", self.device)
        d_rays = torch.from_numpy(rays).to(dev)
        d_idx = torch.empty(n, dtype=torch.int32, device=dev)
        d_t = torch.empty((n, 2), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _native.check(_native.load().rtgs_trace_closest(self.handle, n, d_rays.data_ptr(), d_idx.data_ptr(),
                                                        d_t.data_ptr(), stream))
        idx = d_idx.cpu().numpy()
        depth = np.full(n, -1, np.int32)
        if (idx >= 0).any():
            bf = self.bvh_field.to_numpy()
            inv = np.empty(self._n, np.int64)
            inv[self.read_lbvh()["sorted_idx"]] = np.arange(self._n)
            hitm = idx >= 0
            depth[hitm] = bf["depth"][self._n - 1 + inv[idx[hitm]]]
        return SceneHit(gaussian_idx=idx, intersections=d_t.cpu().numpy(), depth=depth)

    # ------------------------------------------------------------------ arbitrary rays
    def _rays_arg(self, rays):
        """``rays`` as a contiguous, 16-byte aligned CUDA float32 (..., 8) tensor on the scene's device."""
        import torch
        dev = torch.device("cuda", self.device)
        if not isinstance(rays, torch.Tensor) or rays.device != dev or rays.dtype != torch.float32:
            raise ValueError(f"rays: expected a float32 tensor on {dev}")
        if rays.dim() < 1 or rays.shape[-1] != 8:
            raise ValueError(f"rays: expected shape (..., 8), got {tuple(rays.shape)}")
        rays = rays.detach().contiguous()
        if rays.data_ptr() % 16:
            rays = rays.clone()
        return rays

    @staticmethod
    def _buffer(t, shape, name, dev):
        import torch
        if t is None:
            return None
        if (not isinstance(t, torch.Tensor) or t.device != dev or t.dtype != torch.float32
                or tuple(t.shape) != tuple(shape) or not t.is_contiguous()):
            raise ValueError(f"{name}: expected a contiguous float32 tensor of shape {tuple(shape)} on {dev}")
        return t

    def render_rays(self, rays, depth: int = 16, t_cut: float = 0.0, out=None, out_T=None, out_depth=None,
                    with_depth: bool = False):
        """Composite arbitrary rays (rtgs_render_rays) on the current stream and return ``(rgb (..., 3), T (...))``.

        ``rays`` is a CUDA float32 tensor of shape (..., 8) on the scene's device: origin, direction (used as given,
        not normalised), start, end - the record of ``Camera.generate_ray_field``, so a (W,H,8) ray field gives a
        (W,H,3) image in the layout of ``RayTracer.render_device``.  Each ray composites its ``depth`` nearest
        Gaussians with start < t1 < end, front to back while T >= ``t_cut``.  ``out`` / ``out_T`` may pass the output
        tensors.  With ``out_depth`` (...) or ``with_depth=True`` it returns ``(rgb, T, D)``: D = sum_k T_k alpha_k t*_k,
        t*_k the ray parameter (units of the ray's d) of layer k's max-response point (rtgs_render_rays_depth)."""
        import torch
        rays = self._rays_arg(rays)
        dev = rays.device
        lead = tuple(rays.shape[:-1])
        out = self._buffer(out, lead + (3,), "out", dev)
        out_T = self._buffer(out_T, lead, "out_T", dev)
        if out is None:
            out = torch.empty(lead + (3,), dtype=torch.float32, device=dev)
        if out_T is None:
            out_T = torch.empty(lead, dtype=torch.float32, device=dev)
        out_depth = self._buffer(out_depth, lead, "out_depth", dev)
        if out_depth is None and with_depth:
            out_depth = torch.empty(lead, dtype=torch.float32, device=dev)
        head = (self.handle, rays.numel() // 8, rays.data_ptr(), int(depth), float(t_cut), out.data_ptr(),
                out_T.data_ptr())
        stream = torch.cuda.current_stream(dev).cuda_stream
        if out_depth is None:
            _native.check(_native.load().rtgs_render_rays(*head, stream))
            return out, out_T
        _native.check(_native.load().rtgs_render_rays_depth(*head, out_depth.data_ptr(), stream))
        return out, out_T, out_depth

    def render_rays_backward(self, rays, dL_drgb, dL_dT=None, depth: int = 16, t_cut: float = 0.0, grads=None,
                             rays_grad: bool = False, replay: bool = False, dL_dD=None):
        """Gradient of ``render_rays(rays, depth, t_cut)`` with each ray's layer list held fixed
        (rtgs_render_rays_backward), on the current stream.

        dL_drgb (..., 3) and dL_dT (...) are CUDA float32 tensors shaped like the rays.  Returns a dict of (n, ...)
        float32 gradients ``pos rot scale color opacity`` and ``sh`` (scenes with SH), as ``RayTracer.render_backward``
        does; with ``rays_grad=True`` also ``rays`` (..., 8): dL/do in columns 0-2, dL/dd in 3-5, zeros in 6-7.
        ``grads`` may pass tensors of these names to accumulate into (missing ones are zero-initialised).  With
        ``replay=True`` the dict also holds ``rgb`` / ``T``, the image the backward recomputed.  ``dL_dD`` (...) is the
        gradient with respect to the depth of ``render_rays(with_depth=True)`` (rtgs_render_rays_backward_depth); with
        it, ``replay=True`` also returns ``depth``."""
        import torch
        rays = self._rays_arg(rays)
        dev = rays.device
        lead = tuple(rays.shape[:-1])
        dL_drgb = self._buffer(dL_drgb.contiguous(), lead + (3,), "dL_drgb", dev)
        dL_dT = None if dL_dT is None else self._buffer(dL_dT.contiguous(), lead, "dL_dT", dev)
        dL_dD = None if dL_dD is None else self._buffer(dL_dD.contiguous(), lead, "dL_dD", dev)
        n = self._n
        shapes = dict(pos=(n, 3), rot=(n, 4), scale=(n, 3), color=(n, 3), opacity=(n,))
        if self.has_sh:
            shapes["sh"] = (n, 15, 3)
        if rays_grad:
            shapes["rays"] = lead + (8,)
        out = dict(grads or {})
        for name, shape in shapes.items():
            if name not in out:
                out[name] = torch.zeros(shape, dtype=torch.float32, device=dev)
            else:
                self._buffer(out[name], shape, f"grads[{name!r}]", dev)
        if replay:
            out["rgb"] = torch.empty(lead + (3,), dtype=torch.float32, device=dev)
            out["T"] = torch.empty(lead, dtype=torch.float32, device=dev)
            if dL_dD is not None:
                out["depth"] = torch.empty(lead, dtype=torch.float32, device=dev)
        ptr = lambda k: out[k].data_ptr() if k in out else None  # noqa: E731
        args = (self.handle, rays.numel() // 8, rays.data_ptr(), int(depth), float(t_cut), dL_drgb.data_ptr(),
                None if dL_dT is None else dL_dT.data_ptr(), ptr("pos"), ptr("rot"), ptr("scale"), ptr("color"),
                ptr("opacity"), ptr("sh"), ptr("rays") if rays_grad else None, ptr("rgb"), ptr("T"))
        stream = torch.cuda.current_stream(dev).cuda_stream
        if dL_dD is None:
            _native.check(_native.load().rtgs_render_rays_backward(*args, stream))
        else:
            _native.check(_native.load().rtgs_render_rays_backward_depth(*args, dL_dD.data_ptr(), ptr("depth"),
                                                                         stream))
        return out
