"""Differentiable rendering: ``render`` as a ``torch.autograd.Function`` over the Gaussian parameters.

Forward: the parameters are copied into the scene in place (``Scene.set_gaussians``, LBVH rebuilt) and the region is
rendered with ``rtgs_render`` on the current stream.  Backward: ``rtgs_render_backward`` into zero-initialised
gradients.  The gradient is that of the image with each pixel's layer list held fixed (the layers' membership and
order, and the q = 3 silhouette, have none); the camera pose gets none.  A minimal optimisation loop::

    opt = torch.optim.Adam([pos, color, opacity, sh], lr=1e-2)
    for _ in range(steps):
        rgb, T = rtgs.autograd.render(scene, camera, pos, rot, scale, color, opacity, sh)
        loss = ((rgb - target) ** 2).mean(); opt.zero_grad(); loss.backward(); opt.step()

Each call rebuilds the scene's LBVH from the current values (the parameters may have moved since the last step), so
the forward of one step and the backward of the same step see the same tree only if no other call updates the scene
in between.
"""
from __future__ import annotations

import torch

from . import _native
from .ray_tracer import MAX_DEPTH

_NAMES = ("pos", "rot", "scale", "color", "opacity", "sh")


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scene, camera, depth, t_cut, tile, pos, rot, scale, color, opacity, sh):
        params = [t.detach().contiguous() if t is not None else None for t in (pos, rot, scale, color, opacity, sh)]
        scene.set_gaussians(*params)
        dev = torch.device("cuda", scene.device)
        W, H = camera.buf_size.x, camera.buf_size.y
        x0, y0, w, h = (0, 0, W, H) if tile is None else tile
        rgb = torch.empty((w, h, 3), dtype=torch.float32, device=dev)
        T = torch.empty((w, h), dtype=torch.float32, device=dev)
        cam = camera.native()
        _native.check(_native.load().rtgs_render(scene.handle, cam, x0, y0, w, h, int(depth), float(t_cut), 0, 0,
                                                 rgb.data_ptr(), T.data_ptr(),
                                                 torch.cuda.current_stream(dev).cuda_stream, None))
        ctx.scene, ctx.cam, ctx.region, ctx.depth, ctx.t_cut = scene, cam, (x0, y0, w, h), int(depth), float(t_cut)
        ctx.has_sh = sh is not None
        ctx.dev = dev
        return rgb, T

    @staticmethod
    def backward(ctx, g_rgb, g_T):
        scene, dev = ctx.scene, ctx.dev
        x0, y0, w, h = ctx.region
        n = scene.num_gaussians
        shapes = dict(pos=(n, 3), rot=(n, 4), scale=(n, 3), color=(n, 3), opacity=(n,), sh=(n, 15, 3))
        need = dict(zip(_NAMES, ctx.needs_input_grad[5:]))
        need["sh"] = need["sh"] and ctx.has_sh
        grads = {k: torch.zeros(shapes[k], dtype=torch.float32, device=dev) if need[k] else None for k in _NAMES}
        if g_rgb is None:
            g_rgb = torch.zeros((w, h, 3), dtype=torch.float32, device=dev)
        g_rgb = g_rgb.to(torch.float32).contiguous()
        g_T = None if g_T is None else g_T.to(torch.float32).contiguous()
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        _native.check(_native.load().rtgs_render_backward(
            scene.handle, ctx.cam, x0, y0, w, h, ctx.depth, ctx.t_cut, g_rgb.data_ptr(), ptr(g_T),
            *(ptr(grads[k]) for k in _NAMES), None, None, torch.cuda.current_stream(dev).cuda_stream))
        return (None, None, None, None, None) + tuple(grads[k] for k in _NAMES)


def render(scene, camera, pos, rot, scale, color, opacity, sh=None, depth: int = 16, t_cut: float = 0.0, tile=None):
    """Render ``camera`` from the given parameters and return ``(rgb (w,h,3), T (w,h))``, differentiable with respect to
    every parameter tensor that requires a gradient.  The tensors are CUDA float32 on the scene's device with the
    shapes of ``Scene.from_arrays`` (``sh`` iff the scene has SH); the scene's stored parameters become these values.
    ``tile`` = (x0, y0, w, h) restricts the image to a region; layout [i, j] as in ``RayTracer.render_device``."""
    if not 1 <= int(depth) <= MAX_DEPTH:
        raise ValueError(f"depth must be in [1, {MAX_DEPTH}]")
    return _Render.apply(scene, camera, int(depth), float(t_cut), tile, pos, rot, scale, color, opacity, sh)
