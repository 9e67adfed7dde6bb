"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) — float64 reference gradient of the render.

A torch float64 restatement of ``ref_numpy.render`` for small scenes, differentiable with respect to the stored
Gaussian parameters.  The per-pixel layer list (which Gaussians, in which order) is taken from
``ref_numpy.render(..., return_layers=True)`` and held fixed: membership, order and the q = 3 silhouette are piecewise
constant and have no gradient.  Per layer, alpha and the colour are recomputed from the parameters with torch ops:
W = S^-1 Rm^T / |q|^4 exactly as ``local_frame`` (csrc/gsmath.cuh) writes it (Rm = as_rotation_mat3(q), the stored
quaternion used as given), q = |W(o-p) x Wd|^2 / |Wd|^2, alpha = opacity exp(-q), c = colour + sum_j Y_j sh_j.
Compositing is front to back with the renderer's t_cut rule (a layer is composited while the incoming T >= t_cut;
t_cut = 0 is ref_numpy.render).  The gradients are torch autograd's.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ref_numpy as O

NAMES = ("pos", "rot", "scale", "color", "opacity", "sh")


def _rot_mat(q):
    """as_rotation_mat3 (utils/quaternion.py:99-121) of (n,4) xyzw quaternions: (w^2 - |u|^2) I + 2 u u^T + 2 w [u]x."""
    u, w = q[:, :3], q[:, 3]
    a = w * w - (u * u).sum(-1)
    ux, uy, uz = u[:, 0], u[:, 1], u[:, 2]
    z = torch.zeros_like(ux)
    cross = torch.stack([torch.stack([z, -uz, uy], -1), torch.stack([uz, z, -ux], -1),
                         torch.stack([-uy, ux, z], -1)], -2)
    eye = torch.eye(3, dtype=q.dtype)
    return a[:, None, None] * eye + 2.0 * u[:, :, None] * u[:, None, :] + 2.0 * w[:, None, None] * cross


def local_frame(rot, scale):
    """W (n,3,3) with Sigma^-1 = W^T W: W[k][j] = Rm[j][k] / (s_k |q|^4) (csrc/gsmath.cuh local_frame)."""
    Rm = _rot_mat(rot)
    c = (rot * rot).sum(-1)
    return Rm.transpose(1, 2) / (scale[:, :, None] * (c * c)[:, None, None])


def render(gs: O.GaussianSet, cam: O.CameraParams, depth: int = 16, t_cut: float = 0.0, pixels=None, params=None):
    """The image of ``ref_numpy.render`` (plus the t_cut rule) as torch float64 tensors.

    Returns dict(rgb (W,H,3) or (n,3), T, params = the float64 leaf tensors (requires_grad) the image depends on,
    layers = ref_numpy's per-pixel layer list, nlayers = layers composited per pixel after the t_cut rule).
    ``params`` may pass those leaves in."""
    ref = O.render(gs, cam, depth=depth, pixels=pixels, return_layers=True)
    idx = torch.from_numpy(ref["layers"]["idx"].astype(np.int64))          # (R,K), -1 = no layer
    o, dirs = O.camera_rays(cam, pixels)
    o = torch.from_numpy(np.asarray(o, np.float64))
    d = torch.from_numpy(np.asarray(dirs, np.float64))
    if params is None:
        src = dict(pos=gs.pos, rot=gs.rot, scale=gs.scale, color=gs.color, opacity=gs.opacity, sh=gs.sh)
        params = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in src.items()
                  if v is not None}
    W = local_frame(params["rot"], params["scale"])                        # (N,3,3)
    dn = d / torch.linalg.norm(d, dim=-1, keepdim=True)
    Y = torch.from_numpy(O.sh_basis(dn.numpy()))                          # (R,15)
    R, K = idx.shape
    nl = torch.zeros(R, dtype=torch.int64)
    T = torch.ones(R, dtype=torch.float64)
    rgb = torch.zeros((R, 3), dtype=torch.float64)
    for k in range(K):
        g = idx[:, k]
        live = (g >= 0) & (T >= t_cut)
        if not bool(live.any()):
            break
        gg = torch.where(live, g, torch.zeros_like(g))
        Wg = W[gg]
        u = torch.einsum("rij,rj->ri", Wg, o[None, :] - params["pos"][gg])
        v = torch.einsum("rij,rj->ri", Wg, d)
        m = torch.linalg.cross(u, v)
        q = (m * m).sum(-1) / (v * v).sum(-1)
        alpha = torch.where(live, params["opacity"][gg] * torch.exp(-q), torch.zeros_like(q))
        c = params["color"][gg]
        if "sh" in params:
            c = c + torch.einsum("rk,rkc->rc", Y, params["sh"][gg])
        rgb = rgb + (T * alpha)[:, None] * c
        T = T * (1.0 - alpha)
        nl += live.to(torch.int64)
    if pixels is None:
        rgb = rgb.reshape(cam.width, cam.height, 3)
        T = T.reshape(cam.width, cam.height)
    return dict(rgb=rgb, T=T, params=params, layers=ref["layers"], nlayers=nl.numpy())


def grad(gs: O.GaussianSet, cam: O.CameraParams, dL_drgb, dL_dT=None, depth: int = 16, t_cut: float = 0.0,
         pixels=None):
    """Gradients (float64 numpy, original order, shapes of the parameters) of
    L = sum(dL_drgb * rgb) + sum(dL_dT * T), and the image: dict(pos, rot, scale, color, opacity[, sh], rgb, T)."""
    out = render(gs, cam, depth=depth, t_cut=t_cut, pixels=pixels)
    L = (out["rgb"] * torch.as_tensor(np.asarray(dL_drgb, np.float64))).sum()
    if dL_dT is not None:
        L = L + (out["T"] * torch.as_tensor(np.asarray(dL_dT, np.float64))).sum()
    names = [k for k in NAMES if k in out["params"]]
    gr = torch.autograd.grad(L, [out["params"][k] for k in names], allow_unused=True)
    res = {k: (np.zeros(tuple(out["params"][k].shape)) if g is None else g.numpy()) for k, g in zip(names, gr)}
    res["rgb"] = out["rgb"].detach().numpy()
    res["T"] = out["T"].detach().numpy()
    return res
