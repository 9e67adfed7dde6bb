"""Ray tracer Gaussian splatting renderer — mirror of the reference's ``rtgs/ray_tracer.py``.

The reference renders one compositing layer per ``sample()`` call (one full BVH traversal per
pixel per layer, ray / T / accum round-tripping through global memory; ray_tracer.py:39-104).
Here a whole sample — ray generation, one LBVH traversal per 4x8-pixel tile, ``depth`` nearest
entries, front-to-back compositing — is ONE fused CUDA kernel (csrc/render.cu).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native
from .camera import Camera
from .fields import DeviceField
from .scene import Scene
from .utils.types import vec2i

MAX_DEPTH = 32  # RTGS_MAX_DEPTH


class PendingFrame:
    """A frame queued by ``RayTracer.render_async``.  Frames complete in submission order: ``result()``
    first collects every older frame of the same scene."""

    def __init__(self, scene, out):
        self._scene = scene
        self._out = out
        self.done = False

    def result(self):
        pending = self._scene._pending
        while not self.done:
            head = pending[0]
            try:
                _native.check(_native.load().rtgs_render_host_collect(self._scene.handle))
            finally:
                pending.popleft()
                head.done = True
        return self._out


class RayTracer:
    """RayTracer(buf_size, scene, camera) — ray_tracer.py:25-37.

    Buffers (shape (W,H[,3]), origin bottom-left, index [i, j] = [column, row from the bottom]):
    ``sample_buf`` accumulated radiance, ``attenuation_buf`` transmittance T, ``disp_buf`` display.
    ``t_cut`` is the transmittance early-termination threshold (the reference has none; 0 disables)."""

    def __init__(self, buf_size, scene: Scene, camera: Camera, t_cut: float = 1e-4) -> None:
        import torch
        self.scene = scene
        self.camera = camera
        self.buf_size = vec2i(buf_size)
        self.t_cut = float(t_cut)
        dev = torch.device("cuda", scene.device if scene.device is not None else 0)
        self._dev = dev
        W, H = self.buf_size.x, self.buf_size.y
        self.sample_buf = DeviceField(torch.zeros((W, H, 3), dtype=torch.float32, device=dev))
        self.attenuation_buf = DeviceField(torch.zeros((W, H), dtype=torch.float32, device=dev))
        self.disp_buf = DeviceField(torch.zeros((W, H, 3), dtype=torch.float32, device=dev))
        self.num_steps = 0
        self.num_samples = 0
        self.last_stats = None
        self._pinned = None
        self._async_ring = None
        self._async_next = 0

    # ------------------------------------------------------------------ reference API
    def sample(self, depth: int):
        """Accumulate one sample into the sample buffer (ray_tracer.py:39-54).

        Observable state (num_steps / num_samples, final sample_buf) follows the reference's state
        machine: ``depth`` calls make one sample.  The whole sample is rendered by the fused kernel on
        the FIRST call of the sample (num_steps == 0); the remaining calls only advance the counters
        (SURVEY.md §7 hard part 8)."""
        if self.num_steps == 0:
            self._render_into(depth, accumulate=True)
        self.num_steps += 1
        if self.num_steps >= depth:
            self.num_steps = 0
            self.num_samples += 1

    def clear_sample(self):
        """ray_tracer.py:56-60."""
        self.sample_buf.fill(0.0)

    def clear_attenuation(self):
        """ray_tracer.py:62-66."""
        self.attenuation_buf.fill(1.0)

    def generate_disp_buffer(self, num_samples: int, num_steps: int, num_depth: int):
        """ray_tracer.py:68-77: disp = sample_buf / (num_samples + num_steps/num_depth).

        Because a sample is complete after its first ``sample()`` call here, a sample in progress
        (num_steps > 0) counts as a whole one; at sample boundaries (num_steps == 0) the result is the
        reference's."""
        import torch
        denom = float(num_samples) + (1.0 if num_steps > 0 else 0.0)
        if denom <= 0:
            denom = 1.0
        torch.div(self.sample_buf.tensor, denom, out=self.disp_buf.tensor)

    def sample_step(self):
        """ray_tracer.py:79-104 composites ONE layer; the fused kernel has no single-layer mode, so this
        renders the complete sample when called at the start of a sample and is a no-op otherwise."""
        if self.num_steps == 0:
            self._render_into(MAX_DEPTH if getattr(self, "_depth", None) is None else self._depth, accumulate=True)

    # ------------------------------------------------------------------ additive API
    def render(self, depth: int = 16, tile=None, out=None, pinned: bool = True):
        """Render one complete sample of the current camera and return the image as a host ndarray.

        tile = (x0, y0, w, h) restricts the render to a pixel region (returned array is (w,h,3));
        default is the full (W,H,3) frame.  Layout [i, j] (column, row from the bottom); a conventional
        top-left-origin image is ``img.transpose(1, 0, 2)[::-1]``.

        With ``pinned=True`` (default) the image lands in a pinned host buffer owned by this RayTracer
        and reused by the next ``render()`` of the same size (copy it if you need to keep it); the
        frame is copied into it band by band while later bands still render.  For a sweep over many poses
        use ``render_async`` / ``sweep``.  ``out`` may name any float32 (w,h,3) host array
        instead; ``pinned=False`` returns a fresh pageable array."""
        W, H = self.buf_size.x, self.buf_size.y
        x0, y0, w, h = (0, 0, W, H) if tile is None else tile
        if out is None:
            if pinned:
                if self._pinned is None or self._pinned.shape != (w, h, 3):
                    self._pinned = _native.PinnedBuffer((w, h, 3))
                out = self._pinned.view()
            else:
                out = np.empty((w, h, 3), dtype=np.float32)
        elif out.shape != (w, h, 3) or out.dtype != np.float32 or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous float32 array of shape (w, h, 3)")
        cam = self.camera.native()
        self.scene.drain_pending()
        _native.check(_native.load().rtgs_render_host(self.scene.handle, cam, x0, y0, w, h, int(depth), self.t_cut,
                                                      out.ctypes.data, None))
        return out

    def render_async(self, depth: int = 16, tile=None, fmt: str = "f32"):
        """``render()`` without the wait: queue the frame of the CURRENT camera pose and return a
        ``PendingFrame``; its ``result()`` is the (w,h,3) host image.  Two frames may be in flight per
        scene, so in a sweep frame f+1 renders while the tail of frame f crosses PCIe::

            prev = None
            for pose in poses:
                camera.position, camera.rotation = pose
                cur = tracer.render_async(16)
                if prev is not None:
                    use(prev.result())
                prev = cur
            use(prev.result())

        The image lands in one of three pinned buffers owned by this RayTracer, used in turn: a result
        stays valid until the third ``render_async`` after its own.

        ``fmt`` selects an opt-in COMPACT host image (rtgs_render_host_submit_packed): "f32" (default, the parity
        path, (w,h,3) float32), "f16" ((w,h,3) float16, half the bytes) or "rgba8" ((w,h,4) uint8, clipped to [0,1]
        and rounded like the reference's display, a third of the bytes).  The frame is always rendered in float32;
        only what crosses PCIe changes - for viewer loops and for sweeps on many GPUs of one host."""
        W, H = self.buf_size.x, self.buf_size.y
        x0, y0, w, h = (0, 0, W, H) if tile is None else tile
        fmt_id, dtype, ch = _native.PIXEL_FORMATS[fmt]
        ring = self._async_ring
        if not ring or ring[0].shape != (w, h, ch) or ring[0].dtype != np.dtype(dtype):
            self.scene.drain_pending()
            ring = self._async_ring = [_native.PinnedBuffer((w, h, ch), dtype) for _ in range(3)]
            self._async_next = 0
        buf = ring[self._async_next]
        self._async_next = (self._async_next + 1) % len(ring)
        out = buf.view()
        pending = self.scene._pending
        while len(pending) >= 2:          # the library holds two frames at most
            pending[0].result()
        cam = self.camera.native()
        if fmt_id == 0:
            _native.check(_native.load().rtgs_render_host_submit(self.scene.handle, cam, x0, y0, w, h, int(depth),
                                                                 self.t_cut, out.ctypes.data, None))
        else:
            _native.check(_native.load().rtgs_render_host_submit_packed(self.scene.handle, cam, x0, y0, w, h,
                                                                        int(depth), self.t_cut, out.ctypes.data, fmt_id))
        frame = PendingFrame(self.scene, out)
        pending.append(frame)
        return frame

    def sweep(self, poses, depth: int = 16):
        """Render ``poses`` (an iterable of (position, rotation)) through the two-deep pipeline and yield
        ``(index, image)`` in order; the image is valid until the next-but-one iteration."""
        prev = None
        k = -1
        for k, (pos, rot) in enumerate(poses):
            self.camera.position, self.camera.rotation = pos, rot
            cur = self.render_async(depth)
            if prev is not None:
                yield k - 1, prev.result()
            prev = cur
        if prev is not None:
            yield k, prev.result()

    def render_device(self, depth: int = 16, tile=None, out=None, out_T=None, collect_stats: bool = False,
                      out_depth=None):
        """Render into device memory (a torch CUDA tensor) on the current stream; no host copy.  ``out_depth`` (w,h)
        float32 on the device also receives the composited ray distance D (rtgs_render_depth): D / (1 - T) is the
        expected distance along each pixel's ray."""
        import torch
        W, H = self.buf_size.x, self.buf_size.y
        x0, y0, w, h = (0, 0, W, H) if tile is None else tile
        if out is None:
            out = torch.empty((w, h, 3), dtype=torch.float32, device=self._dev)
        if out_depth is not None and (out_depth.device != self._dev or out_depth.dtype != torch.float32
                                      or tuple(out_depth.shape) != (w, h) or not out_depth.is_contiguous()):
            raise ValueError(f"out_depth: expected a contiguous float32 tensor of shape {(w, h)} on {self._dev}")
        stats = _native.rtgs_render_stats() if collect_stats else None
        cam = self.camera.native()
        args = (self.scene.handle, cam, x0, y0, w, h, int(depth), self.t_cut, 0, 0, out.data_ptr(),
                None if out_T is None else out_T.data_ptr())
        tail = (torch.cuda.current_stream(self._dev).cuda_stream, None if stats is None else C.byref(stats))
        if out_depth is None:
            _native.check(_native.load().rtgs_render(*args, *tail))
        else:
            _native.check(_native.load().rtgs_render_depth(*args, out_depth.data_ptr(), *tail))
        if stats is not None:
            self.last_stats = stats.as_dict()
        return out

    def render_backward(self, dL_drgb, dL_dT=None, depth: int = 16, tile=None, grads=None, replay: bool = False,
                        camera: bool = False, dL_dD=None):
        """Gradient of ``render_device(depth, tile)`` (with ``t_cut``) with respect to the stored Gaussian parameters,
        the layer list of every pixel held fixed (rtgs_render_backward), on the current stream.

        dL_drgb (w,h,3) and dL_dT (w,h) are CUDA float32 tensors of the region.  Returns a dict of (n,...) float32
        gradients ``pos rot scale color opacity`` and ``sh`` (scenes with SH): ``grads`` may pass tensors of these
        names to accumulate into (missing ones are zero-initialised).  With ``replay=True`` the dict also holds
        ``rgb`` / ``T``, the image the backward recomputed.  With ``camera=True`` it also holds the gradient with
        respect to the camera (rtgs_render_backward_camera): ``camera_position`` (3,), ``camera_rotation`` (4,, the
        x,y,z,w quaternion as stored) and ``camera_focal`` (2,), which ``grads`` may pass in the same way.
        ``dL_dD`` (w,h) is the gradient with respect to the depth of ``render_device(out_depth=...)``
        (rtgs_render_backward_depth); with it, ``replay=True`` also returns ``depth``."""
        import torch
        W, H = self.buf_size.x, self.buf_size.y
        x0, y0, w, h = (0, 0, W, H) if tile is None else tile
        n = self.scene.num_gaussians

        def region(t, shape, name):
            if t.device != self._dev or t.dtype != torch.float32 or tuple(t.shape) != shape:
                raise ValueError(f"{name}: expected a float32 tensor of shape {shape} on {self._dev}")
            return t.contiguous()

        dL_drgb = region(dL_drgb, (w, h, 3), "dL_drgb")
        dL_dT = None if dL_dT is None else region(dL_dT, (w, h), "dL_dT")
        dL_dD = None if dL_dD is None else region(dL_dD, (w, h), "dL_dD")
        shapes = dict(pos=(n, 3), rot=(n, 4), scale=(n, 3), color=(n, 3), opacity=(n,))
        if self.scene.has_sh:
            shapes["sh"] = (n, 15, 3)
        if camera:
            shapes.update(camera_position=(3,), camera_rotation=(4,), camera_focal=(2,))
        out = dict(grads or {})
        for name, shape in shapes.items():
            if name not in out:
                out[name] = torch.zeros(shape, dtype=torch.float32, device=self._dev)
            elif (out[name].dtype != torch.float32 or tuple(out[name].shape) != shape or not out[name].is_contiguous()
                  or out[name].device != self._dev):
                raise ValueError(f"grads[{name!r}]: expected a contiguous float32 tensor of shape {shape}")
        if replay:
            out["rgb"] = torch.empty((w, h, 3), dtype=torch.float32, device=self._dev)
            out["T"] = torch.empty((w, h), dtype=torch.float32, device=self._dev)
            if dL_dD is not None:
                out["depth"] = torch.empty((w, h), dtype=torch.float32, device=self._dev)
        cam = self.camera.native()
        ptr = lambda k: out[k].data_ptr() if k in out else None  # noqa: E731
        head = (self.scene.handle, cam, x0, y0, w, h, int(depth), self.t_cut, dL_drgb.data_ptr(),
                None if dL_dT is None else dL_dT.data_ptr(), ptr("pos"), ptr("rot"), ptr("scale"), ptr("color"),
                ptr("opacity"), ptr("sh"))
        tail = (ptr("rgb"), ptr("T"), torch.cuda.current_stream(self._dev).cuda_stream)
        lib = _native.load()
        if dL_dD is not None:
            _native.check(lib.rtgs_render_backward_depth(
                *head, ptr("camera_position"), ptr("camera_rotation"), ptr("camera_focal"), *tail[:2],
                dL_dD.data_ptr(), ptr("depth"), tail[2]))
        elif camera:
            _native.check(lib.rtgs_render_backward_camera(
                *head, ptr("camera_position"), ptr("camera_rotation"), ptr("camera_focal"), *tail))
        else:
            _native.check(lib.rtgs_render_backward(*head, *tail))
        return out

    def _render_into(self, depth, accumulate):
        import torch
        if depth > MAX_DEPTH:
            raise ValueError(f"depth {depth} > {MAX_DEPTH} is not supported by the fused kernel")
        self._depth = int(depth)
        W, H = self.buf_size.x, self.buf_size.y
        cam = self.camera.native()
        _native.check(_native.load().rtgs_render(
            self.scene.handle, cam, 0, 0, W, H, int(depth), self.t_cut, 1 if accumulate else 0, 1,
            self.sample_buf.data_ptr(), self.attenuation_buf.data_ptr(),
            torch.cuda.current_stream(self._dev).cuda_stream, None))
