"""The float64 depth reference (tests/ref_depth.py): a closed form for one Gaussian, central finite differences of D
and of a mixed rgb / T / D loss with the layer lists and t_cut stops held fixed (Gaussians, camera, rays), the
translation and direction-scale identities, and the argument checks of the four depth entry points (no GPU needed)."""
import copy
import ctypes

import numpy as np
import pytest

from oracle import ref_grad as RG
from oracle import ref_numpy as O

import ref_depth as RD
import ref_grad_camera as RC
import ref_rays as RR
from test_oracle_grad import _as_f64, _camera, _scene
from test_oracle_grad_camera import _cam64


def test_one_gaussian_closed_form():
    # an anisotropic Gaussian with a non-unit quaternion, one ray with a non-unit direction
    q = np.array([0.3, -0.2, 0.5, 0.9]) * 1.3
    gs = _as_f64(O.GaussianSet(pos=np.array([[0.2, -0.1, -4.0]]), rot=q[None], scale=np.array([[0.6, 0.3, 0.9]]),
                               color=np.array([[0.5, 0.5, 0.5]]), opacity=np.array([0.8]), sh=None))
    o, d = np.array([0.1, 0.0, 0.3]), np.array([0.05, -0.02, -2.0])
    rays = np.concatenate([o, d, [0.0, np.inf]])[None]
    out = RD.render_rays(gs, rays)
    W = RG.local_frame(*(RG.torch.tensor(v) for v in (gs.rot, gs.scale)))[0].numpy()
    Wd, Wv = W @ d, W @ (gs.pos[0] - o)
    tstar = Wv @ Wd / (Wd @ Wd)
    qm = Wv @ Wv - (Wv @ Wd) ** 2 / (Wd @ Wd)
    alpha = gs.opacity[0] * np.exp(-qm)
    assert out["layers"]["idx"][0, 0] == 0 and qm < 3
    t1 = out["layers"]["t1"][0, 0]
    assert 0 < t1 < tstar   # t* = t1 + sqrt((3 - q) / |Wd|^2)
    assert abs(tstar - (t1 + np.sqrt((3 - qm) / (Wd @ Wd)))) <= 1e-12 * tstar
    assert abs(out["D"].item() - alpha * tstar) <= 1e-14 * tstar
    # o + t* d minimises the Mahalanobis distance along the ray
    f = lambda t: np.sum((W @ (o + t * d - gs.pos[0])) ** 2)   # noqa: E731
    assert f(tstar) < min(f(tstar - 1e-4), f(tstar + 1e-4))
    # scaling d by 2 halves t* and D
    rays2 = rays.copy()
    rays2[0, 3:6] *= 2.0
    assert abs(RD.render_rays(gs, rays2)["D"].item() - 0.5 * alpha * tstar) <= 1e-14 * tstar


def test_pixel_depth_is_the_ray_depth_and_unit_camera_depth_is_distance():
    gs = _scene(12, seed=5, sh=True, unit=False)
    cam = _camera(12, 10)
    a = RD.render_pixels(gs, cam)
    b = RD.render_rays(gs, RR.camera_ray_records(cam))
    assert np.array_equal(a["layers"]["idx"], b["layers"]["idx"])
    assert np.abs(a["D"].detach().numpy() - b["D"].detach().numpy()).max() <= 1e-12
    # rgb and T are the existing references'
    rg = RC.render(gs, cam)
    assert np.abs(a["rgb"].detach().numpy() - rg["rgb"].detach().numpy().reshape(-1, 3)).max() <= 1e-13
    assert np.abs(a["T"].detach().numpy() - rg["T"].detach().numpy().reshape(-1)).max() <= 1e-13
    # a unit camera quaternion has |d| = 1: D / (1 - T) is a distance between the nearest and farthest centre's
    D, T = a["D"].detach().numpy(), a["T"].detach().numpy()
    hit = T < 0.99
    assert hit.mean() > 0.3 and (D[hit] > 0).all()
    dist = np.linalg.norm(np.asarray(gs.pos, np.float64) - np.asarray(cam.position, np.float64), axis=1)
    expect = D[hit] / (1 - T[hit])
    assert (expect > dist.min() - 1.0).all() and (expect < dist.max() + 1.0).all()


def _fd(loss, x, h, count=None):
    """Central differences of loss() with respect to the first ``count`` (default all) elements of the contiguous
    float64 array x (perturbed in place)."""
    assert x.flags.c_contiguous
    g = np.zeros(x.size)
    flat = x.reshape(-1)
    for i in range(x.size if count is None else count):
        v = flat[i]
        flat[i] = v + h
        lp = loss()
        flat[i] = v - h
        lm = loss()
        flat[i] = v
        g[i] = (lp - lm) / (2 * h)
    return g.reshape(x.shape)


def _check(name, ana, fd, tol=1e-6):
    err = np.linalg.norm(ana - fd) / max(np.linalg.norm(fd), 1e-30)
    print(name, f"{err:.1e}")
    assert np.linalg.norm(fd) > 0, name
    assert err <= tol, (name, err)


@pytest.mark.parametrize("case", ["depth_only", "mixed", "nosh", "t_cut", "nonunit_cam"])
def test_pixel_depth_gradients_match_central_differences(case):
    gs = _as_f64(_scene(5, seed=11, sh=case != "nosh", unit=case != "t_cut"))
    t_cut = 0.0
    if case == "t_cut":
        gs.opacity[:] = 0.9
        t_cut = 0.05
    cam = _cam64(_camera(8, 6))
    if case == "nonunit_cam":
        cam.rotation = cam.rotation * 1.2
    R = cam.width * cam.height
    rng = np.random.default_rng(1)
    g_D = rng.normal(size=R)
    g_rgb = np.zeros((R, 3)) if case == "depth_only" else rng.normal(size=(R, 3))
    g_T = None if case == "depth_only" else rng.normal(size=R)
    ana = RD.grad_pixels(gs, cam, g_rgb, g_T, g_D, t_cut=t_cut)
    lay, nl = ana["layers"], ana["nlayers"]
    if t_cut > 0:
        assert (ana["T"] < t_cut).any()   # the rule stops some pixel early

    def loss(g=gs, c=cam):
        own = O.render(g, c, depth=16, return_layers=True)["layers"]
        assert np.array_equal(own["idx"], lay["idx"]), "a perturbation changed a layer list"
        out = RD.render_pixels(g, c, t_cut=t_cut, layers=lay)
        assert np.array_equal(out["nlayers"], nl), "a perturbation moved a t_cut stop"
        L = (out["D"].detach().numpy() * g_D).sum() + (out["rgb"].detach().numpy() * g_rgb).sum()
        return L + (0.0 if g_T is None else (out["T"].detach().numpy() * g_T).sum())

    for k in ("pos", "rot", "scale", "opacity") + (() if case == "depth_only" else ("color",)):
        _check(k, ana[k], _fd(loss, getattr(gs, k), 1e-6))
    if case == "mixed":   # the SH coefficients enter the colour only: those of the first Gaussian
        _check("sh", ana["sh"][0], _fd(loss, gs.sh, 1e-6, count=45)[0])
    cam_pos = cam.position
    _check("cam_position", ana["cam_position"], _fd(loss, cam_pos, 1e-6))
    _check("cam_rotation", ana["cam_rotation"], _fd(loss, cam.rotation, 1e-6))
    focal = np.array(cam.focal, np.float64)

    def loss_f():
        c = copy.copy(cam)
        c.focal = (float(focal[0]), float(focal[1]))
        return loss(c=c)

    _check("cam_focal", ana["cam_focal"], _fd(loss_f, focal, 1e-4))


@pytest.mark.parametrize("case", ["depth_only", "mixed", "nosh", "t_cut", "start", "end"])
def test_ray_depth_gradients_match_central_differences(case):
    from test_oracle_rays import _fd_rays
    gs, rays, t_cut = _fd_rays("nonunit" if case in ("depth_only", "mixed") else case)
    R = rays.shape[0]
    rng = np.random.default_rng(3)
    g_D = rng.normal(size=R)
    g_rgb = np.zeros((R, 3)) if case == "depth_only" else rng.normal(size=(R, 3))
    g_T = None if case == "depth_only" else rng.normal(size=R)
    ana = RD.grad_rays(gs, rays, g_rgb, g_T, g_D, t_cut=t_cut)
    lay, nl = ana["layers"], ana["nlayers"]
    if case == "end":   # a t* beyond `end` still counts
        two = (lay["idx"] >= 0).sum(1) >= 1
        assert two.any()

    def per_ray(r=rays, g=gs):
        own = RR.layer_lists(g, r, 16)
        assert np.array_equal(own["idx"], lay["idx"]), "a perturbation changed a layer list"
        out = RD.render_rays(g, r, t_cut=t_cut, layers=lay)
        assert np.array_equal(out["nlayers"], nl), "a perturbation moved a t_cut stop"
        L = out["D"].detach().numpy() * g_D + (out["rgb"].detach().numpy() * g_rgb).sum(1)
        return L + (0.0 if g_T is None else out["T"].detach().numpy() * g_T)

    for name, cols in (("o", range(0, 3)), ("d", range(3, 6))):
        fd = np.zeros((R, 3))
        for j, c in enumerate(cols):
            h = 1e-6 * np.maximum(1.0, np.abs(rays[:, c]))
            rp, rm = rays.copy(), rays.copy()
            rp[:, c] += h
            rm[:, c] -= h
            fd[:, j] = (per_ray(r=rp) - per_ray(r=rm)) / (2 * h)
        _check(name, ana[name], fd)
    for k in ("pos", "rot", "scale"):
        _check(k, ana[k], _fd(lambda: per_ray().sum(), getattr(gs, k), 1e-6))


@pytest.mark.parametrize("sh", [True, False])
def test_translation_and_direction_scale_identities(sh):
    gs = _as_f64(_scene(6, seed=7, sh=sh, unit=False))
    cam = _cam64(_camera(8, 6))
    cam.rotation = cam.rotation * 1.3
    R = cam.width * cam.height
    rng = np.random.default_rng(5)
    for mixed in (False, True):
        g_D = rng.normal(size=R)
        g_rgb = rng.normal(size=(R, 3)) if mixed else np.zeros((R, 3))
        px = RD.grad_pixels(gs, cam, g_rgb, None, g_D)
        scale = np.linalg.norm(px["cam_position"]) + np.linalg.norm(px["pos"])
        if not mixed:   # D depends on o - p only (the colour's SH direction does not move with a translation either)
            assert np.abs(px["cam_position"] + px["pos"].sum(0)).max() <= 1e-10 * scale
        # d scales with |q_cam|^2: q_cam . dL/dq_cam = -2 sum g_D D
        lhs = float(np.dot(cam.rotation, px["cam_rotation"]))
        rhs = -2.0 * float((g_D * px["D"]).sum())
        assert abs(lhs - rhs) <= 1e-10 * (abs(rhs) + np.linalg.norm(px["cam_rotation"]))
        rays = RR.camera_ray_records(cam)
        rays[:, :3] += rng.normal(0, 0.05, (R, 3))
        ry = RD.grad_rays(gs, rays, g_rgb, None, g_D)
        if not mixed:
            assert np.abs(ry["o"].sum(0) + ry["pos"].sum(0)).max() <= 1e-10 * np.abs(ry["o"]).sum()
        per_ray = (ry["d"] * rays[:, 3:6]).sum(1)
        assert np.abs(per_ray + g_D * ry["D"]).max() <= 1e-10 * max(np.abs(g_D * ry["D"]).max(), 1e-30)


def _dummy_scene():
    # never dereferenced: every call below fails an argument check first
    return ctypes.cast(ctypes.create_string_buffer(64), ctypes.c_void_p)


def test_depth_entry_points_validate_without_a_gpu(lib):
    from rtgs import _native
    buf = ctypes.create_string_buffer(1024)
    base = ctypes.addressof(buf)
    a16 = (base + 15) & ~15          # 16-byte aligned host addresses (never read: every call fails a check first)
    s = _dummy_scene()
    cam = _native.make_camera([0, 0, 0], [0, 0, 0, 1], [10, 10], 8, 8)
    bad_cam = _native.make_camera([0, 0, 0], [0, 0, 0, 1], [0, 10], 8, 8)

    def render(scene=s, cam=cam, x0=0, y0=0, w=8, h=8, depth=16, t_cut=0.0, rgb=a16, dep=a16 + 512):
        return lib.rtgs_render_depth(scene, ctypes.byref(cam), x0, y0, w, h, depth, t_cut, 0, 0, rgb, None, dep,
                                     None, None)

    def backward(scene=s, cam=cam, x0=0, y0=0, w=8, h=8, depth=16, t_cut=0.0, rgb=a16, dep=a16 + 512, rep=None):
        return lib.rtgs_render_backward_depth(scene, ctypes.byref(cam), x0, y0, w, h, depth, t_cut, rgb, None,
                                              *([None] * 11), dep, rep, None)

    image_cases = [dict(scene=None), dict(cam=bad_cam), dict(w=0), dict(x0=-1), dict(x0=1), dict(h=9),
                   dict(depth=0), dict(depth=33), dict(t_cut=-0.1), dict(t_cut=1.0), dict(rgb=None),
                   dict(dep=a16 + 514)]
    for call in (render, backward):
        for kw in image_cases + ([dict(rep=a16 + 2)] if call is backward else []):
            assert call(**kw) == -1, (call.__name__, kw)
            assert b"invalid argument" in lib.rtgs_last_error()

    def rays_fwd(scene=s, n=4, rays=a16, depth=16, t_cut=0.0, rgb=a16 + 256, dep=a16 + 512):
        return lib.rtgs_render_rays_depth(scene, n, rays, depth, t_cut, rgb, None, dep, None)

    def rays_bwd(scene=s, n=4, rays=a16, depth=16, t_cut=0.0, rgb=a16 + 256, dep=a16 + 512, rep=None):
        return lib.rtgs_render_rays_backward_depth(scene, n, rays, depth, t_cut, rgb, None, *([None] * 9), dep,
                                                   rep, None)

    ray_cases = [dict(scene=None), dict(n=-1), dict(rays=None), dict(rays=a16 + 4), dict(rays=a16 + 8),
                 dict(rgb=None), dict(rgb=a16 + 258), dict(depth=0), dict(depth=33), dict(t_cut=-0.1),
                 dict(t_cut=1.0), dict(t_cut=float("nan")), dict(dep=a16 + 513)]
    for call in (rays_fwd, rays_bwd):
        for kw in ray_cases + ([dict(rep=a16 + 1)] if call is rays_bwd else []):
            assert call(**kw) == -1, (call.__name__, kw)
            assert b"invalid argument" in lib.rtgs_last_error()
        # with no rays the buffers are not needed, but the scene, depth and t_cut still are
        assert call(scene=None, n=0, rays=None, rgb=None, dep=None) == -1
        assert call(n=0, rays=None, depth=0, rgb=None, dep=None) == -1
