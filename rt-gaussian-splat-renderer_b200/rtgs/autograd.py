"""Differentiable rendering: ``render`` as a ``torch.autograd.Function`` over the Gaussian parameters and the camera.

Forward: the parameters are copied into the scene in place (``Scene.set_gaussians``, LBVH rebuilt) and the region is
rendered with ``rtgs_render`` on the current stream.  Backward: ``rtgs_render_backward`` into zero-initialised
gradients, or ``rtgs_render_backward_camera`` when a camera tensor needs one.  The gradient is that of the image with
each pixel's layer list held fixed (the layers' membership and order, and the q = 3 silhouette, have none).  A minimal
optimisation loop::

    opt = torch.optim.Adam([pos, color, opacity, sh], lr=1e-2)
    for _ in range(steps):
        rgb, T = rtgs.autograd.render(scene, camera, pos, rot, scale, color, opacity, sh)
        loss = ((rgb - target) ** 2).mean(); opt.zero_grad(); loss.backward(); opt.step()

Each call rebuilds the scene's LBVH from the current values (the parameters may have moved since the last step), so
the forward of one step and the backward of the same step see the same tree only if no other call updates the scene
in between.  ``render_camera`` renders the scene as stored, differentiable with respect to the camera only, and
rebuilds nothing: the loop of pose refinement or of tracking a camera against a fixed scene.  ``render_rays`` renders
arbitrary rays (non-pinhole cameras, ray batches drawn from many views) and differentiates with respect to the rays
too (``rtgs_render_rays`` / ``rtgs_render_rays_backward``).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native
from .ray_tracer import MAX_DEPTH

_NAMES = ("pos", "rot", "scale", "color", "opacity", "sh")
_CAM_SHAPES = dict(cam_position=(3,), cam_rotation=(4,), cam_focal=(2,))


def _native_camera(camera, position, rotation, focal):
    """``camera`` as the C struct, with the given float32 tensors in place of its position, rotation and focal
    length (the render takes the camera by value: CUDA tensors are read back, which synchronises)."""
    vals = {}
    for (name, shape), t in zip(_CAM_SHAPES.items(), (position, rotation, focal)):
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or tuple(t.shape) != shape:
            raise ValueError(f"{name}: expected a float32 tensor of shape {shape}")
        vals[name] = np.asarray(t.detach().cpu().numpy(), np.float32)
    return _native.make_camera(vals.get("cam_position", np.asarray(camera.position, np.float32)),
                               vals.get("cam_rotation", np.asarray(camera.rotation, np.float32)),
                               vals.get("cam_focal", np.asarray(camera.focal_length, np.float32)),
                               camera.buf_size.x, camera.buf_size.y)


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scene, camera, depth, t_cut, tile, update, cam_position, cam_rotation, cam_focal,
                pos, rot, scale, color, opacity, sh):
        if update:
            params = [t.detach().contiguous() if t is not None else None
                      for t in (pos, rot, scale, color, opacity, sh)]
            scene.set_gaussians(*params)
        dev = torch.device("cuda", scene.device)
        W, H = camera.buf_size.x, camera.buf_size.y
        x0, y0, w, h = (0, 0, W, H) if tile is None else tile
        rgb = torch.empty((w, h, 3), dtype=torch.float32, device=dev)
        T = torch.empty((w, h), dtype=torch.float32, device=dev)
        cam = _native_camera(camera, cam_position, cam_rotation, cam_focal)
        _native.check(_native.load().rtgs_render(scene.handle, cam, x0, y0, w, h, int(depth), float(t_cut), 0, 0,
                                                 rgb.data_ptr(), T.data_ptr(),
                                                 torch.cuda.current_stream(dev).cuda_stream, None))
        ctx.scene, ctx.cam, ctx.region, ctx.depth, ctx.t_cut = scene, cam, (x0, y0, w, h), int(depth), float(t_cut)
        ctx.has_sh = sh is not None
        ctx.cam_devices = tuple(None if t is None else t.device for t in (cam_position, cam_rotation, cam_focal))
        ctx.dev = dev
        return rgb, T

    @staticmethod
    def backward(ctx, g_rgb, g_T):
        scene, dev = ctx.scene, ctx.dev
        x0, y0, w, h = ctx.region
        n = scene.num_gaussians
        shapes = dict(pos=(n, 3), rot=(n, 4), scale=(n, 3), color=(n, 3), opacity=(n,), sh=(n, 15, 3))
        need = dict(zip(_NAMES, ctx.needs_input_grad[9:]))
        need["sh"] = need["sh"] and ctx.has_sh
        grads = {k: torch.zeros(shapes[k], dtype=torch.float32, device=dev) if need[k] else None for k in _NAMES}
        cam_grads = [torch.zeros(shape, dtype=torch.float32, device=dev) if nd else None
                     for shape, nd in zip(_CAM_SHAPES.values(), ctx.needs_input_grad[6:9])]
        if g_rgb is None:
            g_rgb = torch.zeros((w, h, 3), dtype=torch.float32, device=dev)
        g_rgb = g_rgb.to(torch.float32).contiguous()
        g_T = None if g_T is None else g_T.to(torch.float32).contiguous()
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        lib = _native.load()
        head = (scene.handle, ctx.cam, x0, y0, w, h, ctx.depth, ctx.t_cut, g_rgb.data_ptr(), ptr(g_T),
                *(ptr(grads[k]) for k in _NAMES))
        tail = (None, None, torch.cuda.current_stream(dev).cuda_stream)
        if any(g is not None for g in cam_grads):
            _native.check(lib.rtgs_render_backward_camera(*head, *(ptr(g) for g in cam_grads), *tail))
        else:
            _native.check(lib.rtgs_render_backward(*head, *tail))
        cam_grads = [None if g is None else g.to(d) for g, d in zip(cam_grads, ctx.cam_devices)]
        return (None,) * 6 + tuple(cam_grads) + tuple(grads[k] for k in _NAMES)


def render(scene, camera, pos, rot, scale, color, opacity, sh=None, depth: int = 16, t_cut: float = 0.0, tile=None, *,
           cam_position=None, cam_rotation=None, cam_focal=None):
    """Render ``camera`` from the given parameters and return ``(rgb (w,h,3), T (w,h))``, differentiable with respect to
    every parameter tensor that requires a gradient.  The tensors are CUDA float32 on the scene's device with the
    shapes of ``Scene.from_arrays`` (``sh`` iff the scene has SH); the scene's stored parameters become these values.
    ``tile`` = (x0, y0, w, h) restricts the image to a region; layout [i, j] as in ``RayTracer.render_device``.

    ``cam_position`` (3,), ``cam_rotation`` (4,, x,y,z,w, used as given like ``Camera.rotation``) and ``cam_focal``
    (2,) are optional float32 tensors on any device that replace the camera's values for this call and receive
    gradients when they require them (each on its own device).  The render takes the camera by value, so their
    values are read to the host in the forward: CUDA tensors cost one synchronisation."""
    if not 1 <= int(depth) <= MAX_DEPTH:
        raise ValueError(f"depth must be in [1, {MAX_DEPTH}]")
    return _Render.apply(scene, camera, int(depth), float(t_cut), tile, True, cam_position, cam_rotation, cam_focal,
                         pos, rot, scale, color, opacity, sh)


def render_camera(scene, camera, position=None, rotation=None, focal=None, depth: int = 16, t_cut: float = 0.0,
                  tile=None):
    """Render the scene as stored and return ``(rgb (w,h,3), T (w,h))``, differentiable with respect to the camera
    only: ``position`` (3,), ``rotation`` (4,) and ``focal`` (2,) are float32 tensors as in ``render`` (their values
    are read to the host in the forward, one synchronisation for CUDA tensors); the ones left None are the camera's.
    The scene is neither updated nor rebuilt, which makes this the step of pose refinement or tracking::

        opt = torch.optim.Adam([position, rotation], lr=1e-3)
        for _ in range(steps):
            rgb, _ = rtgs.autograd.render_camera(scene, camera, position, rotation)
            loss = ((rgb - target) ** 2).mean(); opt.zero_grad(); loss.backward(); opt.step()
    """
    if not 1 <= int(depth) <= MAX_DEPTH:
        raise ValueError(f"depth must be in [1, {MAX_DEPTH}]")
    return _Render.apply(scene, camera, int(depth), float(t_cut), tile, False, position, rotation, focal,
                         None, None, None, None, None, None)


class _RenderRays(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scene, depth, t_cut, update, rays, pos, rot, scale, color, opacity, sh):
        if update:
            scene.set_gaussians(*(t.detach().contiguous() if t is not None else None
                                  for t in (pos, rot, scale, color, opacity, sh)))
        rgb, T = scene.render_rays(rays, depth, t_cut)
        ctx.save_for_backward(rays)
        ctx.scene, ctx.depth, ctx.t_cut, ctx.has_sh = scene, depth, t_cut, sh is not None
        return rgb, T

    @staticmethod
    def backward(ctx, g_rgb, g_T):
        (rays,) = ctx.saved_tensors
        scene = ctx.scene
        rays_c = scene._rays_arg(rays)
        dev, lead = rays_c.device, tuple(rays_c.shape[:-1])
        n = scene.num_gaussians
        shapes = dict(pos=(n, 3), rot=(n, 4), scale=(n, 3), color=(n, 3), opacity=(n,), sh=(n, 15, 3))
        need = dict(zip(_NAMES, ctx.needs_input_grad[5:]))
        need["sh"] = need["sh"] and ctx.has_sh
        grads = {k: torch.zeros(shapes[k], dtype=torch.float32, device=dev) if need[k] else None for k in _NAMES}
        g_rays = torch.zeros(lead + (8,), dtype=torch.float32, device=dev) if ctx.needs_input_grad[4] else None
        if g_rgb is None:
            g_rgb = torch.zeros(lead + (3,), dtype=torch.float32, device=dev)
        g_rgb = g_rgb.to(torch.float32).contiguous()
        g_T = None if g_T is None else g_T.to(torch.float32).contiguous()
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        _native.check(_native.load().rtgs_render_rays_backward(
            scene.handle, rays_c.numel() // 8, rays_c.data_ptr(), ctx.depth, ctx.t_cut, g_rgb.data_ptr(), ptr(g_T),
            *(ptr(grads[k]) for k in _NAMES), ptr(g_rays), None, None, torch.cuda.current_stream(dev).cuda_stream))
        return (None,) * 4 + (g_rays,) + tuple(grads[k] for k in _NAMES)


def render_rays(scene, rays, pos=None, rot=None, scale=None, color=None, opacity=None, sh=None, depth: int = 16,
                t_cut: float = 0.0):
    """Composite arbitrary rays and return ``(rgb (..., 3), T (...))``, differentiable with respect to the rays and,
    when they are given, the Gaussian parameters (``Scene.render_rays`` / ``render_rays_backward``).

    ``rays`` is a CUDA float32 (..., 8) tensor on the scene's device (origin, direction, start, end); it gets a
    gradient (dL/do, dL/dd; none for start and end) when it requires one, so any camera model written in torch is
    differentiable through the render.  Pass either every Gaussian tensor (``sh`` iff the scene has SH), and the
    scene is updated and rebuilt from them as in ``render``, or none, and the stored scene is rendered as it is:
    nothing is rebuilt and nothing is read to the host.  A training step on random rays of many views::

        rays = torch.cat([cam_rays[v][idx[v]] for v in views])          # (B, 8)
        rgb, _ = rtgs.autograd.render_rays(scene, rays, pos, rot, scale, color, opacity, sh)
        loss = ((rgb - target) ** 2).mean(); opt.zero_grad(); loss.backward(); opt.step()
    """
    if not 1 <= int(depth) <= MAX_DEPTH:
        raise ValueError(f"depth must be in [1, {MAX_DEPTH}]")
    given = [t is not None for t in (pos, rot, scale, color, opacity)]
    if any(given) and not all(given):
        raise ValueError("pass all of pos, rot, scale, color, opacity (and sh for a scene with SH), or none")
    if not any(given) and sh is not None:
        raise ValueError("sh was given without the other Gaussian tensors")
    return _RenderRays.apply(scene, int(depth), float(t_cut), all(given), rays, pos, rot, scale, color, opacity, sh)
