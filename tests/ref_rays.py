"""TEST INFRASTRUCTURE ONLY — the float64 reference render and gradient for arbitrary rays.

A ray is the (8,) record of ``rtgs_generate_rays``: origin o, direction d (used as given, not normalised), start, end.
Its layer list is computed with the local-frame test of ``exact_intersect`` (csrc/gsmath.cuh): u = W(o - p), v = W d,
q = |u x v|^2 / |v|^2, a hit iff |v|^2 (3 - q) > 0, the near root t1 = (-u.v - sqrt(|v|^2 (3 - q))) / |v|^2; the hits
with start < t1 < end, sorted by ascending t1 (ties by Gaussian index), truncated to ``depth``.  The compositing is
``oracle.ref_grad``'s (alpha = opacity exp(-q), c = colour + sum_j Y_j(d/|d|) sh_j, front to back under the t_cut
rule), in torch float64 with the Gaussian parameters and the per-ray o and d as leaves.  A ray with a non-finite o or
d component, d = 0 or !(start < end) composites nothing (rgb 0, T 1).  ``layers=`` holds another call's lists fixed,
so that finite differences differentiate the image with the lists held fixed, as the kernels do.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import ref_grad as RG
from oracle import ref_numpy as O

import ref_grad_camera as RC

RAY_NAMES = ("o", "d")


def valid_rays(rays):
    """(R,) bool: the rays that composite anything."""
    rays = np.asarray(rays, np.float64).reshape(-1, 8)
    finite = np.isfinite(rays[:, :6]).all(1)
    with np.errstate(invalid="ignore"):
        return finite & (np.abs(rays[:, 3:6]).sum(1) > 0) & (rays[:, 6] < rays[:, 7])


def layer_lists(gs: O.GaussianSet, rays, depth: int = 16, chunk: int = 512):
    """Per ray the ``depth`` nearest hits with start < t1 < end: dict(idx (R,K) int, -1 padded; t1 (R,K))."""
    rays = np.asarray(rays, np.float64).reshape(-1, 8)
    R, K = rays.shape[0], int(depth)
    W = RG.local_frame(torch.tensor(np.asarray(gs.rot, np.float64)),
                       torch.tensor(np.asarray(gs.scale, np.float64))).numpy()      # (N,3,3)
    p = np.asarray(gs.pos, np.float64)
    ok = valid_rays(rays)
    idx = np.full((R, K), -1, np.int64)
    tt = np.full((R, K), np.inf)
    for s in range(0, R, chunk):
        e = min(R, s + chunk)
        o, d = rays[s:e, :3], rays[s:e, 3:6]
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            u = np.einsum("nij,rnj->rni", W, o[:, None, :] - p[None, :, :])
            v = np.einsum("nij,rj->rni", W, d)
            A = (v * v).sum(-1)
            m = np.cross(u, v)
            q = (m * m).sum(-1) / A
            disc = A * (3.0 - q)
            t1 = (-(u * v).sum(-1) - np.sqrt(np.where(disc > 0, disc, 0.0))) / A
            keep = (disc > 0) & (t1 > rays[s:e, 6:7]) & (t1 < rays[s:e, 7:8]) & ok[s:e, None]
        t1 = np.where(keep, t1, np.inf)
        order = np.argsort(t1, axis=1, kind="stable")[:, :K]
        ts = np.take_along_axis(t1, order, axis=1)
        kk = order.shape[1]
        idx[s:e, :kk] = np.where(np.isfinite(ts), order, -1)
        tt[s:e, :kk] = ts
    return dict(idx=idx, t1=tt)


def render(gs: O.GaussianSet, rays, depth: int = 16, t_cut: float = 0.0, layers=None):
    """The image of the rays (R,8) as torch float64 tensors from float64 leaves of the Gaussian parameters and of the
    per-ray o (R,3) and d (R,3).  Returns dict(rgb (R,3), T (R,), params, layers, nlayers = layers composited per ray
    after the t_cut rule)."""
    rays = np.asarray(rays, np.float64).reshape(-1, 8)
    if layers is None:
        layers = layer_lists(gs, rays, depth)
    idx = torch.from_numpy(layers["idx"].astype(np.int64))
    ok = torch.from_numpy(valid_rays(rays))
    src = dict(pos=gs.pos, rot=gs.rot, scale=gs.scale, color=gs.color, opacity=gs.opacity, sh=gs.sh)
    params = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in src.items() if v is not None}
    # degenerate rays keep their leaves, but compute on a harmless stand-in: they have no layers
    safe = np.where(valid_rays(rays)[:, None], rays[:, :6], np.array([0.0, 0.0, 0.0, 0.0, 0.0, 1.0]))
    params["o"] = torch.tensor(rays[:, :3].copy(), requires_grad=True)
    params["d"] = torch.tensor(rays[:, 3:6].copy(), requires_grad=True)
    o = torch.where(ok[:, None], params["o"], torch.from_numpy(safe[:, :3]))
    d = torch.where(ok[:, None], params["d"], torch.from_numpy(safe[:, 3:6]))
    W = RG.local_frame(params["rot"], params["scale"])
    Y = RC.sh_basis(d / torch.linalg.norm(d, dim=-1, keepdim=True))
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
        u = torch.einsum("rij,rj->ri", Wg, o - params["pos"][gg])
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
    return dict(rgb=rgb, T=T, params=params, layers=layers, nlayers=nl.numpy())


def grad(gs: O.GaussianSet, rays, dL_drgb, dL_dT=None, depth: int = 16, t_cut: float = 0.0, layers=None):
    """Gradients (float64 numpy) of L = sum(dL_drgb * rgb) + sum(dL_dT * T) with respect to the Gaussian parameters
    (original order, their shapes) and the rays (o (R,3), d (R,3)), and the image:
    dict(pos, rot, scale, color, opacity[, sh], o, d, rgb, T, layers, nlayers)."""
    out = render(gs, rays, depth=depth, t_cut=t_cut, layers=layers)
    L = (out["rgb"] * torch.as_tensor(np.asarray(dL_drgb, np.float64).reshape(-1, 3))).sum()
    if dL_dT is not None:
        L = L + (out["T"] * torch.as_tensor(np.asarray(dL_dT, np.float64).reshape(-1))).sum()
    names = [k for k in RG.NAMES + RAY_NAMES if k in out["params"]]
    gr = torch.autograd.grad(L, [out["params"][k] for k in names], allow_unused=True)
    res = {k: (np.zeros(tuple(out["params"][k].shape)) if g is None else g.numpy()) for k, g in zip(names, gr)}
    res["rgb"] = out["rgb"].detach().numpy()
    res["T"] = out["T"].detach().numpy()
    res["layers"], res["nlayers"] = out["layers"], out["nlayers"]
    return res


def camera_ray_records(cam: O.CameraParams, pixels=None):
    """``ref_numpy.camera_rays`` as (R,8) float64 records with start 0 and end +inf."""
    o, d = O.camera_rays(cam, pixels)
    rays = np.zeros((d.shape[0], 8))
    rays[:, :3] = o
    rays[:, 3:6] = d
    rays[:, 7] = np.inf
    return rays
