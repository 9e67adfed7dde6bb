"""The float64 reference for arbitrary rays (tests/ref_rays.py): the image against the pixel oracles, the ray
gradient chained through the camera model against the camera gradient, central finite differences with the layer
lists held fixed, and the argument checks of rtgs_render_rays / rtgs_render_rays_backward (no GPU needed)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_grad as RG
from oracle import ref_numpy as O

import ref_grad_camera as RC
import ref_rays as RR
from test_oracle_grad import _as_f64, _camera, _scene
from test_oracle_grad_camera import _cam64


@pytest.mark.parametrize("sh", [True, False])
@pytest.mark.parametrize("depth", [1, 3, 16])
def test_camera_rays_render_the_pixel_oracles(sh, depth):
    gs = _scene(12, seed=3 + depth, sh=sh, unit=False)
    cam = _camera(12, 10)
    rays = RR.camera_ray_records(cam)
    got = RR.render(gs, rays, depth=depth)
    want = O.render(gs, cam, depth=depth, return_layers=True)
    rg = RG.render(gs, cam, depth=depth)
    assert np.array_equal(got["layers"]["idx"], want["layers"]["idx"])
    rgb, T = got["rgb"].detach().numpy(), got["T"].detach().numpy()
    e1 = np.abs(rgb - want["rgb"].reshape(-1, 3)).max()
    e2 = np.abs(rgb - rg["rgb"].detach().numpy().reshape(-1, 3)).max()
    e3 = np.abs(T - want["T"].reshape(-1)).max()
    print(f"ref_numpy {e1:.1e}, ref_grad {e2:.1e}, T {e3:.1e}")
    assert max(e1, e2, e3) <= 1e-12
    assert (want["nhit"] > 0).mean() > 0.5


@pytest.mark.parametrize("sh", [True, False])
def test_ray_gradient_chained_through_the_camera_is_the_camera_gradient(sh):
    gs = _as_f64(_scene(6, seed=11, sh=sh, unit=False))
    cam = _cam64(_camera(8, 6))
    cam.rotation = cam.rotation * 1.2   # a non-unit camera quaternion: |d| = 1.44
    rng = np.random.default_rng(2)
    g_rgb = rng.normal(size=(cam.width * cam.height, 3))
    g_T = rng.normal(size=cam.width * cam.height)
    want = RC.grad(gs, cam, g_rgb.reshape(cam.width, cam.height, 3), g_T.reshape(cam.width, cam.height), depth=16)
    leaves = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True)
              for k, v in (("position", cam.position), ("rotation", cam.rotation),
                           ("focal", [float(cam.focal[0]), float(cam.focal[1])]))}
    o, d = RC.camera_rays(cam, leaves["position"], leaves["rotation"], leaves["focal"])
    rays = np.zeros((d.shape[0], 8))
    rays[:, :3] = o.detach().numpy()
    rays[:, 3:6] = d.detach().numpy()
    rays[:, 7] = np.inf
    got = RR.grad(gs, rays, g_rgb, g_T, depth=16)
    o_b = o.expand_as(d)
    chained = torch.autograd.grad([o_b, d], list(leaves.values()),
                                  [torch.from_numpy(got["o"]), torch.from_numpy(got["d"])])
    for (name, g), k in zip(zip(leaves, chained), RC.CAM_NAMES):
        err = np.linalg.norm(g.numpy() - want[k]) / np.linalg.norm(want[k])
        print(name, f"{err:.1e}")
        assert err <= 1e-10, (name, err)
    for k in RG.NAMES:   # and the Gaussian gradients are the pixel path's
        if k in want:
            assert np.linalg.norm(got[k] - want[k]) <= 1e-10 * np.linalg.norm(want[k]), k


def _fd_rays(case):
    """Rays of a small view for a finite-difference case, the scene and the t_cut."""
    sh = case != "nosh"
    gs = _as_f64(_scene(5, seed=11, sh=sh, unit=case not in ("nonunit", "t_cut")))   # t_cut: test_oracle_grad's scene
    t_cut = 0.0
    if case == "t_cut":
        gs.opacity[:] = 0.9
        t_cut = 0.05
    rays = RR.camera_ray_records(_camera(8, 6))
    rng = np.random.default_rng(4)
    # move the origins off the camera centre so that the rays do not share one
    rays[:, :3] += rng.normal(0, 0.05, (rays.shape[0], 3))
    if case == "unit":
        rays[:, 3:6] /= np.linalg.norm(rays[:, 3:6], axis=1, keepdims=True)
    else:
        rays[:, 3:6] *= rng.uniform(0.3, 3.0, (rays.shape[0], 1))
    lay = RR.layer_lists(gs, rays, 16)
    n = (lay["idx"] >= 0).sum(1)
    t = lay["t1"]
    if case == "start":
        two = n >= 2   # start between the first two hits drops the nearest layer
        rays[two, 6] = 0.5 * (t[two, 0] + t[two, 1])
    if case == "end":
        two = n >= 2   # end between the first two hits drops every layer but the nearest
        rays[two, 7] = 0.5 * (t[two, 0] + t[two, 1])
    return gs, rays, t_cut


@pytest.mark.parametrize("case", ["unit", "nonunit", "nosh", "t_cut", "start", "end"])
def test_ray_gradients_match_central_differences(case):
    gs, rays, t_cut = _fd_rays(case)
    R = rays.shape[0]
    rng = np.random.default_rng(1)
    g_rgb = rng.normal(size=(R, 3))
    g_T = rng.normal(size=R)
    ana = RR.grad(gs, rays, g_rgb, g_T, depth=16, t_cut=t_cut)
    base = RR.render(gs, rays, depth=16, t_cut=t_cut)
    if case in ("start", "end"):
        full = rays.copy()
        full[:, 6], full[:, 7] = 0.0, np.inf
        dropped = (RR.layer_lists(gs, full, 16)["idx"] >= 0).sum() - (base["layers"]["idx"] >= 0).sum()
        assert dropped > 0, "the interval drops no layer"
    if t_cut > 0:
        assert (base["T"].detach().numpy() < t_cut).any()   # the rule stops some ray early

    def per_ray_loss(r):
        own = RR.layer_lists(gs, r, 16)
        assert np.array_equal(own["idx"], base["layers"]["idx"]), "a perturbation changed a layer list"
        out = RR.render(gs, r, depth=16, t_cut=t_cut, layers=base["layers"])
        assert np.array_equal(out["nlayers"], base["nlayers"]), "a perturbation moved a t_cut stop"
        return (out["rgb"].detach().numpy() * g_rgb).sum(1) + out["T"].detach().numpy() * g_T

    # rays are independent: one perturbation of component c of every ray gives every ray's derivative
    for name, cols in (("o", range(0, 3)), ("d", range(3, 6))):
        fd = np.zeros((R, 3))
        for j, c in enumerate(cols):
            h = 1e-6 * np.maximum(1.0, np.abs(rays[:, c]))
            rp, rm = rays.copy(), rays.copy()
            rp[:, c] += h
            rm[:, c] -= h
            fd[:, j] = (per_ray_loss(rp) - per_ray_loss(rm)) / (2 * h)
        err = np.linalg.norm(ana[name] - fd) / max(np.linalg.norm(fd), 1e-30)
        print(case, name, f"{err:.1e}")
        assert np.linalg.norm(fd) > 0, name
        assert err <= 1e-6, (name, err)
    # scaling d changes neither q nor the order of t1 nor d / |d|
    dot = (ana["d"] * rays[:, 3:6]).sum(1)
    assert np.abs(dot).max() <= 1e-9 * np.linalg.norm(ana["d"]) * np.linalg.norm(rays[:, 3:6])


def test_degenerate_rays_composite_nothing():
    gs = _scene(5, seed=11)
    rays = RR.camera_ray_records(_camera(8, 6))
    rays[0, 0] = np.nan
    rays[1, 4] = np.inf
    rays[2, 3:6] = 0.0
    rays[3, 6] = rays[3, 7] = 1.0
    rays[4, 7] = np.nan
    R = rays.shape[0]
    out = RR.grad(gs, rays, np.ones((R, 3)), np.ones(R))
    assert list(RR.valid_rays(rays)) == [False] * 5 + [True] * (R - 5)
    assert (out["T"][5:] < 1).any()
    assert (out["rgb"][:5] == 0).all() and (out["T"][:5] == 1).all()
    assert (out["o"][:5] == 0).all() and (out["d"][:5] == 0).all()


def _dummy_scene():
    # never dereferenced: every call below fails an argument check first
    return ctypes.cast(ctypes.create_string_buffer(64), ctypes.c_void_p)


def test_ray_entry_points_validate_without_a_gpu(lib):
    buf = ctypes.create_string_buffer(1024)
    base = ctypes.addressof(buf)
    a16 = (base + 15) & ~15          # 16-byte aligned host addresses (never read: every call fails a check first)
    s = _dummy_scene()

    def fwd(scene=s, n=4, rays=a16, depth=16, t_cut=0.0, rgb=a16 + 256):
        return lib.rtgs_render_rays(scene, n, rays, depth, t_cut, rgb, None, None)

    def bwd(scene=s, n=4, rays=a16, depth=16, t_cut=0.0, dl=a16 + 256):
        return lib.rtgs_render_rays_backward(scene, n, rays, depth, t_cut, dl, None, *([None] * 9), None)

    for call in (fwd, bwd):
        rgb_kw = "rgb" if call is fwd else "dl"
        cases = [dict(scene=None), dict(n=-1), dict(rays=None), dict(rays=a16 + 4), dict(rays=a16 + 8),
                 {rgb_kw: None}, {rgb_kw: a16 + 258}, dict(depth=0), dict(depth=33), dict(t_cut=-0.1),
                 dict(t_cut=1.0), dict(t_cut=float("nan"))]
        for kw in cases:
            assert call(**kw) == -1, (call.__name__, kw)
            assert b"invalid argument" in lib.rtgs_last_error()
        # with no rays the buffers are not needed, but the scene, depth and t_cut still are
        assert call(scene=None, n=0, rays=None, **{rgb_kw: None}) == -1
        assert call(n=0, rays=None, depth=0, **{rgb_kw: None}) == -1
