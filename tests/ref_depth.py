"""TEST INFRASTRUCTURE ONLY — the float64 reference of the depth image (rtgs_render_depth / rtgs_render_rays_depth).

For a ray (o, d) with composited layers k (the layer lists and the t_cut rule of ``oracle.ref_grad``,
``ref_grad_camera`` and ``ref_rays``, held fixed by passing ``layers``):

    t*_k = (p - o)^T W^T W d / |W d|^2        the ray parameter of layer k's max-response point (units of d)
    D    = sum_k T_k alpha_k t*_k            composited like one more colour channel, not normalised

with W = local_frame as rendered (``oracle.ref_grad.local_frame``, non-unit stored quaternions as given).  The pixel
form takes the Gaussian parameters and the camera (position, rotation, focal) as float64 torch leaves, the ray form
the Gaussian parameters and each ray's o and d.  A degenerate ray has no layers: D = 0.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import ref_grad as RG
from oracle import ref_numpy as O

import ref_grad_camera as RC
import ref_rays as RR


def _composite(params, o, d, idx, t_cut):
    """rgb (R,3), T (R,), D (R,), the layers composited per ray (front to back under the t_cut rule) and the largest
    composited |t*| per ray (the scale of D's tolerances).
    o is (3,) or (R,3), d (R,3), idx (R,K) with -1 = no layer."""
    W = RG.local_frame(params["rot"], params["scale"])
    Y = RC.sh_basis(d / torch.linalg.norm(d, dim=-1, keepdim=True))
    o = o.expand_as(d)
    R, K = idx.shape
    nl = torch.zeros(R, dtype=torch.int64)
    T = torch.ones(R, dtype=torch.float64)
    D = torch.zeros(R, dtype=torch.float64)
    tmax = torch.zeros(R, dtype=torch.float64)
    rgb = torch.zeros((R, 3), dtype=torch.float64)
    for k in range(K):
        g = idx[:, k]
        live = (g >= 0) & (T >= t_cut)
        if not bool(live.any()):
            break
        gg = torch.where(live, g, torch.zeros_like(g))
        Wg = W[gg]
        u = torch.einsum("rij,rj->ri", Wg, o - params["pos"][gg])
        v = torch.einsum("rij,rj->ri", Wg, d)
        A = (v * v).sum(-1)
        m = torch.linalg.cross(u, v)
        q = (m * m).sum(-1) / A
        tstar = -(u * v).sum(-1) / A
        alpha = torch.where(live, params["opacity"][gg] * torch.exp(-q), torch.zeros_like(q))
        c = params["color"][gg]
        if "sh" in params:
            c = c + torch.einsum("rk,rkc->rc", Y, params["sh"][gg])
        w = T * alpha
        rgb = rgb + w[:, None] * c
        D = D + w * tstar
        tmax = torch.maximum(tmax, torch.where(live, tstar.detach().abs(), torch.zeros_like(tmax)))
        T = T * (1.0 - alpha)
        nl += live.to(torch.int64)
    return rgb, T, D, nl.numpy(), tmax.numpy()


def render_pixels(gs: O.GaussianSet, cam: O.CameraParams, depth: int = 16, t_cut: float = 0.0, pixels=None,
                  layers=None):
    """The pixels of ``cam`` (all, (W,H) order, or ``pixels``) as flat (R,...) torch float64 tensors:
    dict(rgb, T, D, params = Gaussian and camera leaves (ref_grad_camera names), layers, nlayers, tmax)."""
    if layers is None:
        layers = O.render(gs, cam, depth=depth, pixels=pixels, return_layers=True)["layers"]
    src = dict(pos=gs.pos, rot=gs.rot, scale=gs.scale, color=gs.color, opacity=gs.opacity, sh=gs.sh,
               cam_position=cam.position, cam_rotation=cam.rotation,
               cam_focal=[float(cam.focal[0]), float(cam.focal[1])])
    params = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in src.items() if v is not None}
    o, d = RC.camera_rays(cam, params["cam_position"], params["cam_rotation"], params["cam_focal"], pixels)
    idx = torch.from_numpy(layers["idx"].astype(np.int64))
    rgb, T, D, nl, tmax = _composite(params, o, d, idx, t_cut)
    return dict(rgb=rgb, T=T, D=D, params=params, layers=layers, nlayers=nl, tmax=tmax)


def render_rays(gs: O.GaussianSet, rays, depth: int = 16, t_cut: float = 0.0, layers=None):
    """The rays (R,8) as torch float64 tensors: dict(rgb, T, D, params = Gaussian leaves and o, d, layers, nlayers)."""
    rays = np.asarray(rays, np.float64).reshape(-1, 8)
    if layers is None:
        layers = RR.layer_lists(gs, rays, depth)
    ok = torch.from_numpy(RR.valid_rays(rays))
    src = dict(pos=gs.pos, rot=gs.rot, scale=gs.scale, color=gs.color, opacity=gs.opacity, sh=gs.sh)
    params = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in src.items() if v is not None}
    # degenerate rays keep their leaves but compute on a harmless stand-in: they have no layers
    safe = torch.tensor([0.0, 0.0, 0.0, 0.0, 0.0, 1.0], dtype=torch.float64)
    params["o"] = torch.tensor(rays[:, :3].copy(), requires_grad=True)
    params["d"] = torch.tensor(rays[:, 3:6].copy(), requires_grad=True)
    o = torch.where(ok[:, None], params["o"], safe[:3])
    d = torch.where(ok[:, None], params["d"], safe[3:])
    idx = torch.from_numpy(layers["idx"].astype(np.int64))
    rgb, T, D, nl, tmax = _composite(params, o, d, idx, t_cut)
    return dict(rgb=rgb, T=T, D=D, params=params, layers=layers, nlayers=nl, tmax=tmax)


def _grad(out, names, g_rgb, g_T, g_D):
    L = (out["rgb"] * torch.as_tensor(np.asarray(g_rgb, np.float64).reshape(-1, 3))).sum()
    if g_T is not None:
        L = L + (out["T"] * torch.as_tensor(np.asarray(g_T, np.float64).reshape(-1))).sum()
    if g_D is not None:
        L = L + (out["D"] * torch.as_tensor(np.asarray(g_D, np.float64).reshape(-1))).sum()
    names = [k for k in names if k in out["params"]]
    gr = torch.autograd.grad(L, [out["params"][k] for k in names], allow_unused=True)
    res = {k: (np.zeros(tuple(out["params"][k].shape)) if g is None else g.numpy()) for k, g in zip(names, gr)}
    for k in ("rgb", "T", "D"):
        res[k] = out[k].detach().numpy()
    res["layers"], res["nlayers"], res["tmax"] = out["layers"], out["nlayers"], out["tmax"]
    return res


def grad_pixels(gs, cam, g_rgb, g_T=None, g_D=None, depth: int = 16, t_cut: float = 0.0, pixels=None, layers=None):
    """Gradients (float64 numpy) of L = sum(g_rgb rgb) + sum(g_T T) + sum(g_D D) over the pixels with respect to the
    Gaussian parameters and the camera, and the flat images: dict(pos, ..., cam_focal, rgb, T, D, layers, nlayers)."""
    out = render_pixels(gs, cam, depth=depth, t_cut=t_cut, pixels=pixels, layers=layers)
    return _grad(out, RG.NAMES + RC.CAM_NAMES, g_rgb, g_T, g_D)


def grad_rays(gs, rays, g_rgb, g_T=None, g_D=None, depth: int = 16, t_cut: float = 0.0, layers=None):
    """Gradients (float64 numpy) of the same loss over rays with respect to the Gaussian parameters and the rays'
    o (R,3) and d (R,3), and the images: dict(pos, ..., o, d, rgb, T, D, layers, nlayers)."""
    out = render_rays(gs, rays, depth=depth, t_cut=t_cut, layers=layers)
    return _grad(out, RG.NAMES + RR.RAY_NAMES, g_rgb, g_T, g_D)
