"""TEST INFRASTRUCTURE ONLY — the float64 reference gradient of the render with respect to the camera.

``oracle.ref_grad.render`` with the camera position, quaternion and focal length as float64 torch leaves as well:
the rays are ``ref_numpy.camera_rays`` restated in torch (px = (i + 0.5 - W/2) / fx, dc = n / |n|, d = q dc q* with the
stored quaternion used as given, not normalised, as ref_numpy does), and the compositing is ``oracle.ref_grad``'s
(W = S^-1 Rm^T / |q|^4, q = |W(o-p) x Wd|^2 / |Wd|^2, alpha = opacity exp(-q), c = colour + sum_j Y_j(d/|d|) sh_j,
front to back with the t_cut rule).  The per-pixel layer lists are ref_numpy's for ``cam``, or the ``layers`` passed
in, e.g. those of an unperturbed camera, so that finite differences hold them fixed.  The gradients are torch
autograd's.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import ref_grad as RG
from oracle import ref_numpy as O

CAM_NAMES = ("cam_position", "cam_rotation", "cam_focal")


def sh_basis(dirs):
    """ref_numpy.sh_basis (the `5z^2 - 3z` term as coded) of a torch (n,3) tensor of normalised directions."""
    x, y, z = dirs[..., 0], dirs[..., 1], dirs[..., 2]
    return torch.stack([
        0.5 * O.C0 * y,
        0.5 * O.C0 * z,
        0.5 * O.C0 * x,
        0.5 * O.C1 * x * y,
        0.5 * O.C1 * y * z,
        0.25 * O.C2 * (3 * z ** 2 - 1),
        0.5 * O.C1 * x * z,
        0.25 * O.C1 * (x ** 2 - y ** 2),
        0.25 * O.C3 * y * (3 * x ** 2 - y ** 2),
        0.5 * O.C4 * x * y * z,
        0.25 * O.C5 * y * (5 * z ** 2 - 1),
        0.25 * O.C6 * (5 * z ** 2 - 3 * z),
        0.25 * O.C5 * x * (5 * z ** 2 - 1),
        0.25 * O.C4 * (x ** 2 - y ** 2) * z,
        0.25 * O.C3 * x * (x ** 2 - 3 * y ** 2),
    ], -1)


def _quat_mul(p, q):
    """ref_numpy.quat_mul (utils/quaternion.py:8-23) of xyzw quaternions, broadcasting."""
    pv, pw, qv, qw = p[..., :3], p[..., 3:4], q[..., :3], q[..., 3:4]
    w = pw * qw - (pv * qv).sum(-1, keepdim=True)
    pv, qv = torch.broadcast_tensors(pv, qv)
    v = pw * qv + qw * pv + torch.linalg.cross(pv, qv)
    return torch.cat([v, w], -1)


def camera_rays(cam: O.CameraParams, position, rotation, focal, pixels=None):
    """``ref_numpy.camera_rays`` in torch float64: (origin (3,), dirs (n,3)) from the ``position`` (3,), ``rotation``
    (4,) and ``focal`` (2,) tensors, differentiable with respect to them."""
    W, H = cam.width, cam.height
    if pixels is None:
        ii, jj = np.meshgrid(np.arange(W), np.arange(H), indexing="ij")
        pixels = np.stack([ii.ravel(), jj.ravel()], axis=-1)
    pixels = np.asarray(pixels)
    u = torch.from_numpy((pixels[:, 0] + 0.5) / W)                         # camera.py:68-70
    v = torch.from_numpy((pixels[:, 1] + 0.5) / H)
    px = (W * u - 0.5 * W) / focal[0]                                      # camera.py:46-47
    py = (H * v - 0.5 * H) / focal[1]
    dc = torch.stack([px, py, -torch.ones_like(px)], -1)
    dc = dc / torch.linalg.norm(dc, dim=-1, keepdim=True)                  # camera.py:49-50
    qv = torch.cat([dc, torch.zeros_like(dc[:, :1])], -1)
    conj = rotation * torch.tensor([-1.0, -1.0, -1.0, 1.0], dtype=torch.float64)
    d = _quat_mul(rotation[None, :], _quat_mul(qv, conj[None, :]))[:, :3]  # camera.py:52 (rot_vec3)
    return position, d


def render(gs: O.GaussianSet, cam: O.CameraParams, depth: int = 16, t_cut: float = 0.0, pixels=None, layers=None):
    """The image of ``ref_numpy.render`` (plus the t_cut rule) as torch float64 tensors, from float64 leaves of the
    Gaussian parameters and of the camera (float64 copies of ``cam``'s position, rotation and focal length).

    Returns dict(rgb (W,H,3) or (n,3), T, params = the leaves (Gaussian names of oracle.ref_grad, and CAM_NAMES),
    layers = the per-pixel layer lists used, nlayers = layers composited per pixel after the t_cut rule).
    ``layers`` (the ``layers`` of an earlier result) replaces ref_numpy's lists for ``cam``."""
    if layers is None:
        layers = O.render(gs, cam, depth=depth, pixels=pixels, return_layers=True)["layers"]
    idx = torch.from_numpy(layers["idx"].astype(np.int64))                 # (R,K), -1 = no layer
    src = dict(pos=gs.pos, rot=gs.rot, scale=gs.scale, color=gs.color, opacity=gs.opacity, sh=gs.sh,
               cam_position=cam.position, cam_rotation=cam.rotation,
               cam_focal=[float(cam.focal[0]), float(cam.focal[1])])
    params = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in src.items() if v is not None}
    o, d = camera_rays(cam, params["cam_position"], params["cam_rotation"], params["cam_focal"], pixels)
    W = RG.local_frame(params["rot"], params["scale"])                     # (N,3,3)
    Y = sh_basis(d / torch.linalg.norm(d, dim=-1, keepdim=True))           # (R,15)
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
    return dict(rgb=rgb, T=T, params=params, layers=layers, nlayers=nl.numpy())


def grad(gs: O.GaussianSet, cam: O.CameraParams, dL_drgb, dL_dT=None, depth: int = 16, t_cut: float = 0.0,
         pixels=None, layers=None):
    """Gradients (float64 numpy) of L = sum(dL_drgb * rgb) + sum(dL_dT * T) with respect to the Gaussian parameters
    (original order, their shapes) and the camera (cam_position (3,), cam_rotation (4,), cam_focal (2,)), and the
    image: dict(pos, rot, scale, color, opacity[, sh], cam_position, cam_rotation, cam_focal, rgb, T)."""
    out = render(gs, cam, depth=depth, t_cut=t_cut, pixels=pixels, layers=layers)
    L = (out["rgb"] * torch.as_tensor(np.asarray(dL_drgb, np.float64))).sum()
    if dL_dT is not None:
        L = L + (out["T"] * torch.as_tensor(np.asarray(dL_dT, np.float64))).sum()
    names = [k for k in RG.NAMES + CAM_NAMES if k in out["params"]]
    gr = torch.autograd.grad(L, [out["params"][k] for k in names], allow_unused=True)
    res = {k: (np.zeros(tuple(out["params"][k].shape)) if g is None else g.numpy()) for k, g in zip(names, gr)}
    res["rgb"] = out["rgb"].detach().numpy()
    res["T"] = out["T"].detach().numpy()
    return res
