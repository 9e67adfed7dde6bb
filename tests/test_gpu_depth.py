"""Depth rendering on the GPU (rtgs_render_depth, rtgs_render_rays_depth and their backward passes): RGB and T
bit-identical to the plain calls, D bit-identical across every render route, D and its gradients against the float64
reference (tests/ref_depth.py), the translation and direction-scale identities, the NULL-depth calls as their
counterparts, the output contract (regions, full-image pitch, stripes, accumulate) and rtgs.autograd."""
import numpy as np
import pytest

from oracle import ref_numpy as O

import ref_depth as RD
from gpu_util import make_camera, make_scene, random_set
from test_gpu_backward import ATOMIC_TOL, GRAD_TOL, GROUPS, _rel, _setup
from test_gpu_rays import _dev, _ray_set, _scene_of

pytestmark = pytest.mark.gpu

DEPTH_TOL = 1e-5      # |D - D_ref| relative to the ray's largest composited t*
IDENTITY_TOL = 1e-5


# ---- scenes of test_gpu_shade_record.py and test_gpu_backward.py ------------------------------------------------
def _cam(pos, rot, W, H, fov):
    from rtgs.camera import Camera
    from rtgs.orbit import focal_from_fov
    f = focal_from_fov(H, fov)
    return Camera(pos, rot, (W, H), (f, f)), O.CameraParams(np.asarray(pos), np.asarray(rot), W, H, (f, f))


def _thin(shape):
    rng = np.random.default_rng(7 if shape == "needles" else 8)
    n = 1500
    pos = rng.uniform(-1, 1, (n, 3))
    pos[:, 2] *= 0.05
    scale = np.full((n, 3), 1.5e-3)
    if shape == "needles":
        scale[np.arange(n), rng.integers(0, 3, n)] = 0.15
    else:
        scale[:, :2] = 0.15 * rng.uniform(0.5, 1.5, (n, 2))
    gs = O.GaussianSet(pos=pos, rot=np.tile([1.0, 0.0, 0.0, 0.0], (n, 1)), scale=scale,
                       color=rng.uniform(0, 1, (n, 3)), opacity=rng.uniform(0.2, 0.99, n),
                       sh=rng.normal(0, 0.15, (n, 15, 3)))
    return gs, *make_camera(0.6, np.pi / 2, 2.5, 120, 80, fov=40.0), 16, 0.0


def _outside_large():
    gs = random_set(2427, seed=11020, mean_scale=0.24913786492941115, sh=True)
    gs.pos[:, 2] *= 0.02
    return gs, *make_camera(2.52281928787616, 2.007240515427329, 0.25061865417331775, 96, 68, fov=31.5), 16, 0.0


def _fov(fov):
    from rtgs.orbit import orbit_pose
    gs = random_set(3000, seed=23, mean_scale=0.04 if fov > 100 else 0.004)
    pos, rot = orbit_pose(1.1, 1.3, 0.6 if fov > 100 else 2.5)
    return gs, *_cam(pos, rot, 97, 70, fov), 16, 0.0


def _qscale(qs):
    from rtgs.orbit import orbit_pose
    gs = random_set(2500, seed=29, mean_scale=0.04)
    pos, rot = orbit_pose(2.2, 1.0, 2.3)
    return gs, *_cam(pos, np.asarray(rot, np.float64) * qs, 88, 72, 55.0), 16, 0.0


def _random(depth, t_cut=0.0, n=1500, seed=13):
    gs = random_set(n, seed=seed, mean_scale=0.08, sh=True)
    if t_cut > 0:
        gs.opacity[:] = np.maximum(gs.opacity, 0.6)
    return gs, *make_camera(0.4, 1.1, 2.6, 64, 48), depth, t_cut


SCENES = {
    "needles": lambda: _thin("needles"),
    "pancakes": lambda: _thin("pancakes"),
    "outside_large": _outside_large,
    "fov170": lambda: _fov(170.0),
    "fov1": lambda: _fov(1.0),
    "qscale0.6": lambda: _qscale(0.6),
    "qscale1.7": lambda: _qscale(1.7),
    "sh_depth16": lambda: _random(16),
    "t_cut_1e-2": lambda: _random(16, t_cut=1e-2),
    "sh_depth32": lambda: _random(32),
}

# (name, scene options) of the render routes; heavy_limit 24 sends every group to the heavy path
ROUTES = [("mode0", dict(render_mode=0)), ("mode2", dict(render_mode=2)), ("mode1", dict(render_mode=1)),
          ("small_pool", dict(render_mode=0, list_pool_chunks=64)),
          ("heavy_fused", dict(render_mode=0, heavy_limit=24, heavy_lists=0)),
          ("heavy_lists1", dict(render_mode=0, heavy_limit=24, heavy_lists=1)),
          ("heavy_lists2", dict(render_mode=0, heavy_limit=24, heavy_lists=2))]
DEFAULTS = dict(render_mode=0, list_pool_chunks=-1, heavy_limit=-1, heavy_lists=0)


def _render(scene, cam, depth, t_cut, with_depth, tile=None, accumulate=0, full=0, out=None):
    """rtgs_render / rtgs_render_depth into fresh (or the given) buffers: (rgb, T, D or None)."""
    import torch
    from rtgs import _native
    dev = torch.device("cuda", scene.device)
    W, H = cam.buf_size.x, cam.buf_size.y
    x0, y0, w, h = (0, 0, W, H) if tile is None else tile
    shape = (W, H) if full else (w, h)
    rgb, T, D = out if out is not None else (torch.empty(shape + (3,), device=dev), torch.empty(shape, device=dev),
                                             torch.empty(shape, device=dev) if with_depth else None)
    lib = _native.load()
    args = (scene.handle, cam.native(), x0, y0, w, h, depth, t_cut, accumulate, full, rgb.data_ptr(), T.data_ptr())
    st = torch.cuda.current_stream(dev).cuda_stream
    if with_depth:
        _native.check(lib.rtgs_render_depth(*args, D.data_ptr(), st, None))
    else:
        _native.check(lib.rtgs_render(*args, st, None))
    torch.cuda.synchronize()
    return rgb, T, D


def _oracle_check(D, T, ref, what):
    """D (flat, float32) against the float64 reference; pixels whose T already differs from the reference's beyond
    rounding (a float32 list that differs from the float64 one) are excluded and counted."""
    D, T = np.asarray(D, np.float64).reshape(-1), np.asarray(T, np.float64).reshape(-1)
    Dr, Tr, tmax = ref["D"].detach().numpy(), ref["T"].detach().numpy(), ref["tmax"]
    keep = np.abs(T - Tr) <= 1e-5
    err = np.abs(D - Dr)[keep] / np.maximum(tmax[keep], 1e-30)
    worst = float(err.max()) if err.size else 0.0
    print(f"{what}: max |D - D_ref| / t*_max {worst:.1e}, excluded {int((~keep).sum())} of {keep.size}")
    assert keep.mean() >= 0.99, what
    assert worst <= DEPTH_TOL, what
    return worst


@pytest.mark.parametrize("name", list(SCENES))
def test_routes_keep_rgb_and_T_and_agree_on_depth(name):
    import torch
    from rtgs.ray_tracer import RayTracer
    gs, cam, ocam, depth, t_cut = SCENES[name]()
    scene = make_scene(gs)
    Ds = {}
    for route, opts in ROUTES:
        for k, v in dict(DEFAULTS, **opts).items():
            scene.set_option(k, v)
        for _ in range(2 if route == "heavy_lists1" else 1):   # mode 1 lists heavy groups once the scene has shown some
            rgb, T, _ = _render(scene, cam, depth, t_cut, False)
            rgb2, T2, D = _render(scene, cam, depth, t_cut, True)
        assert torch.equal(rgb, rgb2) and torch.equal(T, T2), route
        Ds[route] = D
    for k, v in DEFAULTS.items():
        scene.set_option(k, v)
    for route, D in Ds.items():
        assert torch.equal(D, Ds["mode0"]), route
    with torch.no_grad():
        ref = RD.render_pixels(gs, ocam, depth=depth, t_cut=t_cut)
    _oracle_check(Ds["mode0"].cpu().numpy(), T.cpu().numpy(), ref, name)
    # the backward's float64 replay of the same pixels
    rt = RayTracer(cam.buf_size, scene, cam, t_cut=t_cut)
    W, H = cam.buf_size.x, cam.buf_size.y
    z = torch.zeros((W, H), device=rt._dev)
    rep = rt.render_backward(torch.zeros((W, H, 3), device=rt._dev), depth=depth, replay=True, dL_dD=z)
    torch.cuda.synchronize()
    _oracle_check(rep["depth"].cpu().numpy(), rep["T"].cpu().numpy(), ref, name + " replay")
    keep = (np.abs(T.cpu().numpy() - rep["T"].cpu().numpy()) <= 1e-5).reshape(-1)
    diff = np.abs(Ds["mode0"].cpu().numpy() - rep["depth"].cpu().numpy()).reshape(-1)[keep]
    assert (diff <= DEPTH_TOL * np.maximum(ref["tmax"][keep], 1e-30)).all()


def test_output_contract_regions_pitch_stripes_accumulate():
    import torch
    from rtgs.sharding import stripe_columns
    gs = random_set(4000, seed=12, mean_scale=0.03)
    scene = make_scene(gs)
    cam, _ = make_camera(0.9, 1.2, 2.4, 200, 72)
    for depth in (16, 20):
        rgb, T, D = _render(scene, cam, depth, 0.0, True)
        assert (D > 0).any()
        tile = (13, 7, 45, 37)
        _, _, Dr = _render(scene, cam, depth, 0.0, True, tile=tile)
        assert torch.equal(Dr, D[13:58, 7:44])
        # full-image pitch: the region lands at its full-image index, nothing else is touched
        out = (torch.full_like(rgb, -7.0), torch.full_like(T, -7.0), torch.full_like(D, -7.0))
        _render(scene, cam, depth, 0.0, True, tile=tile, full=1, out=out)
        mask = torch.zeros_like(D, dtype=torch.bool)
        mask[13:58, 7:44] = True
        assert torch.equal(out[2][mask], D[mask]) and (out[2][~mask] == -7.0).all()
        # accumulate: out_depth += D, as out_rgb
        acc = (torch.full_like(rgb, 0.25), torch.empty_like(T), torch.full_like(D, 1.5))
        _render(scene, cam, depth, 0.0, True, accumulate=1, out=acc)
        assert torch.equal(acc[2], 1.5 + D) and torch.equal(acc[0], 0.25 + rgb)
        # stripes of three ranks into one buffer
        buf = (torch.empty_like(rgb), torch.empty_like(T), torch.full_like(D, -7.0))
        for r in range(3):
            scene.set_stripe(3, r)
            _render(scene, cam, depth, 0.0, True, full=1, out=buf)
            cols = torch.from_numpy(stripe_columns(200, r, 3)).cuda()
            assert torch.equal(buf[2][cols], D[cols])
        scene.set_stripe()
        assert torch.equal(buf[2], D)


RAY_SCENES = ["axis", "sh_depth16", "nosh_depth4", "sh_depth32", "inside", "nonunit_quaternions", "t_cut_1e-2",
              "single"]


@pytest.mark.parametrize("case", RAY_SCENES)
def test_ray_depth_matches_the_reference_and_the_replay(case):
    import torch
    s = _scene_of(case)
    rays_np = _ray_set(s)
    rays = _dev(rays_np, s)
    rgb, T = s["scene"].render_rays(rays, depth=s["depth"], t_cut=s["t_cut"])
    rgb2, T2, D = s["scene"].render_rays(rays, depth=s["depth"], t_cut=s["t_cut"], with_depth=True)
    R = rays_np.shape[0]
    rep = s["scene"].render_rays_backward(rays, torch.zeros((R, 3), device=s["dev"]), depth=s["depth"],
                                          t_cut=s["t_cut"], replay=True, dL_dD=torch.zeros(R, device=s["dev"]))
    torch.cuda.synchronize()
    assert torch.equal(rgb, rgb2) and torch.equal(T, T2)
    assert torch.equal(rep["depth"], D) and torch.equal(rep["rgb"], rgb) and torch.equal(rep["T"], T)
    with torch.no_grad():
        ref = RD.render_rays(s["gs"], rays_np.astype(np.float64), depth=s["depth"], t_cut=s["t_cut"])
    _oracle_check(D.cpu().numpy(), T.cpu().numpy(), ref, case)
    # a degenerate ray composites nothing
    bad = rays_np[:4].copy()
    bad[0, 0] = np.nan
    bad[1, 3:6] = 0.0
    bad[2, 6] = bad[2, 7] = 1.0
    bad[3, 7] = np.nan
    _, _, Db = s["scene"].render_rays(_dev(bad, s), depth=s["depth"], with_depth=True)
    assert (Db == 0).all()


GRAD_CASES = ["axis", "sh_depth16", "nosh_depth4", "sh_depth32", "ragged_tile", "inside", "nonunit_quaternions",
              "t_cut_1e-2"]


@pytest.mark.parametrize("loss", ["depth_only", "mixed"])
@pytest.mark.parametrize("case", GRAD_CASES)
def test_pixel_gradients_match_the_reference(case, loss):
    import torch
    s = _setup(case)
    x0, y0, w, h = s["region"]
    rng = np.random.default_rng(9)
    g_D = rng.normal(size=(w, h))
    mixed = loss == "mixed"
    g_rgb = s["g_rgb"] if mixed else np.zeros((w, h, 3))
    d_rgb = s["d_rgb"] if mixed else torch.zeros((w, h, 3), device=s["rt"]._dev)
    got = s["rt"].render_backward(d_rgb, s["d_T"] if mixed else None, depth=s["depth"], tile=s["tile"], camera=True,
                                  dL_dD=torch.tensor(g_D, dtype=torch.float32, device=s["rt"]._dev), replay=True)
    torch.cuda.synchronize()
    ii, jj = np.meshgrid(np.arange(x0, x0 + w), np.arange(y0, y0 + h), indexing="ij")
    pixels = np.stack([ii.ravel(), jj.ravel()], -1)
    ref = RD.grad_pixels(s["gs"], s["ocam"], g_rgb.reshape(-1, 3), s["g_T"].reshape(-1) if mixed else None,
                         g_D.reshape(-1), depth=s["depth"], t_cut=s["t_cut"], pixels=pixels)
    assert np.abs(got["depth"].cpu().numpy().reshape(-1) - ref["D"]).max() <= DEPTH_TOL * max(ref["tmax"].max(), 1)
    errs = {}
    for k in GROUPS + ("cam_position", "cam_rotation", "cam_focal"):
        gk = "camera_" + k[4:] if k.startswith("cam_") else k
        if k == "sh" and s["gs"].sh is None:
            continue
        if k in ("color", "sh") and not mixed:
            assert not got[gk].abs().any(), k   # the depth does not depend on the colour
            continue
        assert np.linalg.norm(ref[k]) > 0, k
        errs[k] = _rel(got[gk].cpu().numpy(), ref[k])
    print(case, loss, {k: f"{v:.1e}" for k, v in errs.items()})
    assert max(errs.values()) <= GRAD_TOL, errs
    # identities: D depends on o - p only; d scales with |q_cam|^2 and the rest of the image does not
    D = got["depth"].cpu().numpy().astype(np.float64)
    q = np.asarray(s["cam"].rotation, np.float64)
    lhs = float(np.dot(q, got["camera_rotation"].cpu().numpy()))
    rhs = -2.0 * float((g_D * D).sum())
    assert abs(lhs - rhs) <= IDENTITY_TOL * (abs(rhs) + 1e-3 * np.linalg.norm(ref["cam_rotation"]))
    if not mixed:
        gp = got["camera_position"].cpu().numpy()
        assert np.linalg.norm(gp + got["pos"].sum(0).cpu().numpy()) <= IDENTITY_TOL * np.linalg.norm(gp)


@pytest.mark.parametrize("loss", ["depth_only", "mixed"])
@pytest.mark.parametrize("case", ["axis", "sh_depth16", "nosh_depth4", "inside", "nonunit_quaternions",
                                  "t_cut_1e-2", "single"])
def test_ray_gradients_match_the_reference(case, loss):
    import torch
    s = _scene_of(case)
    rays_np = _ray_set(s, n=1024, seed=2)
    R = rays_np.shape[0]
    rng = np.random.default_rng(3)
    g_D = rng.normal(size=R)
    mixed = loss == "mixed"
    g_rgb = rng.normal(size=(R, 3)) if mixed else np.zeros((R, 3))
    g_T = rng.normal(size=R) if mixed else None
    got = s["scene"].render_rays_backward(_dev(rays_np, s), _dev(g_rgb, s), None if g_T is None else _dev(g_T, s),
                                          depth=s["depth"], t_cut=s["t_cut"], rays_grad=True, replay=True,
                                          dL_dD=_dev(g_D, s))
    torch.cuda.synchronize()
    ref = RD.grad_rays(s["gs"], rays_np.astype(np.float64), g_rgb, g_T, g_D, depth=s["depth"], t_cut=s["t_cut"])
    errs = {}
    for k in GROUPS + ("o", "d"):
        if k == "sh" and s["gs"].sh is None or (k in ("color", "sh") and not mixed):
            continue
        g = got["rays"][:, :3] if k == "o" else got["rays"][:, 3:6] if k == "d" else got[k]
        assert np.linalg.norm(ref[k]) > 0, k
        errs[k] = _rel(g.cpu().numpy(), ref[k])
    print(case, loss, {k: f"{v:.1e}" for k, v in errs.items()})
    assert max(errs.values()) <= GRAD_TOL, errs
    gd = got["rays"][:, 3:6].cpu().numpy().astype(np.float64)
    per_ray = (gd * rays_np[:, 3:6]).sum(1)
    want = -g_D * got["depth"].cpu().numpy()
    scale = np.abs(want).max() + 1e-3 * np.abs(gd * rays_np[:, 3:6]).sum(1).max()
    assert np.abs(per_ray - want).max() <= IDENTITY_TOL * scale
    if not mixed:
        go = got["rays"][:, :3].sum(0).cpu().numpy()
        assert np.linalg.norm(go + got["pos"].sum(0).cpu().numpy()) <= IDENTITY_TOL * np.linalg.norm(go)


def test_null_depth_calls_are_their_counterparts_and_gradients_are_deterministic():
    import torch
    from rtgs import _native
    s = _setup("sh_depth16")
    rt, dev, lib = s["rt"], s["rt"]._dev, _native.load()
    x0, y0, w, h = s["region"]
    n = s["scene"].num_gaussians
    st = torch.cuda.current_stream(dev).cuda_stream
    g_D = torch.randn((w, h), device=dev)

    def pixel(fn, dL_dD=None):
        gr = [torch.zeros(sh, device=dev) for sh in ((n, 3), (n, 4), (n, 3), (n, 3), (n,), (n, 15, 3))]
        cg = [torch.zeros(sh, device=dev) for sh in ((3,), (4,), (2,))]
        args = (s["scene"].handle, rt.camera.native(), x0, y0, w, h, 16, 0.0, s["d_rgb"].data_ptr(),
                s["d_T"].data_ptr(), *(g.data_ptr() for g in gr), *(g.data_ptr() for g in cg), None, None)
        if fn == "camera":
            _native.check(lib.rtgs_render_backward_camera(*args, st))
        else:
            _native.check(lib.rtgs_render_backward_depth(*args, None if dL_dD is None else dL_dD.data_ptr(), None,
                                                         st))
        torch.cuda.synchronize()
        return gr, cg

    a, b = pixel("camera"), pixel("depth")
    assert all(torch.equal(x, y) for x, y in zip(a[1], b[1]))
    assert all(_rel(x.cpu().numpy(), y.cpu().numpy()) <= ATOMIC_TOL for x, y in zip(a[0], b[0]))
    c, d = pixel("depth", g_D), pixel("depth", g_D)
    assert all(torch.equal(x, y) for x, y in zip(c[1], d[1]))
    assert not all(torch.equal(x, y) for x, y in zip(a[1], c[1]))   # the depth term changed the camera gradient

    sr = _scene_of("sh_depth16")
    rays = _dev(_ray_set(sr, n=1024), sr)
    R = rays.shape[0]
    g, gT, gd = torch.randn((R, 3), device=dev), torch.randn(R, device=dev), torch.randn(R, device=dev)

    def ray(fn, dL_dD=None):
        gr = [torch.zeros(sh, device=dev) for sh in ((n, 3), (n, 4), (n, 3), (n, 3), (n,), (n, 15, 3))]
        gray = torch.zeros((R, 8), device=dev)
        args = (sr["scene"].handle, R, rays.data_ptr(), 16, 0.0, g.data_ptr(), gT.data_ptr(),
                *(x.data_ptr() for x in gr), gray.data_ptr(), None, None)
        if fn == "plain":
            _native.check(lib.rtgs_render_rays_backward(*args, st))
        else:
            _native.check(lib.rtgs_render_rays_backward_depth(*args, None if dL_dD is None else dL_dD.data_ptr(),
                                                              None, st))
        torch.cuda.synchronize()
        return gr, gray

    a, b = ray("plain"), ray("depth")
    assert torch.equal(a[1], b[1])
    assert all(_rel(x.cpu().numpy(), y.cpu().numpy()) <= ATOMIC_TOL for x, y in zip(a[0], b[0]))
    c, d = ray("depth", gd), ray("depth", gd)
    assert torch.equal(c[1], d[1]) and not torch.equal(a[1], c[1])


def test_autograd_with_depth_in_all_three_functions(monkeypatch):
    import torch
    import rtgs.autograd as A
    from rtgs import _native
    from rtgs.scene import Scene
    s = _setup("sh_depth16")
    rt, scene, dev = s["rt"], s["scene"], s["rt"]._dev
    W, H = s["region"][2:]
    gv = scene.read_gaussians()
    p = {k: torch.tensor(v, device=dev, requires_grad=True) for k, v in gv.items() if v is not None}
    g_D = torch.randn((W, H), device=dev)
    rgb, T, D = A.render(scene, s["cam"], *(p[k] for k in GROUPS), with_depth=True)
    Dd = torch.empty((W, H), device=dev)
    rgb0 = rt.render_device(16, out_depth=Dd)
    assert torch.equal(D, Dd) and torch.equal(rgb, rgb0)
    (D * g_D).sum().backward()
    direct = rt.render_backward(torch.zeros((W, H, 3), device=dev), dL_dD=g_D)
    for k in GROUPS:
        assert _rel(p[k].grad.cpu().numpy(), direct[k].cpu().numpy()) <= ATOMIC_TOL or not direct[k].abs().any(), k
    # D unused: the plain backward, the same gradients as without with_depth
    for t in p.values():
        t.grad = None
    rgb, T, D = A.render(scene, s["cam"], *(p[k] for k in GROUPS), with_depth=True)
    (rgb * s["d_rgb"]).sum().backward()
    g1 = {k: p[k].grad.clone() for k in GROUPS}
    for t in p.values():
        t.grad = None
    rgb, T = A.render(scene, s["cam"], *(p[k] for k in GROUPS))
    (rgb * s["d_rgb"]).sum().backward()
    for k in GROUPS:
        assert _rel(p[k].grad.cpu().numpy(), g1[k].cpu().numpy()) <= ATOMIC_TOL, k
    # the camera: position and rotation gradients from a depth loss equal the direct call's
    pos = torch.tensor(np.asarray(s["cam"].position, np.float32), requires_grad=True)
    rot = torch.tensor(np.asarray(s["cam"].rotation, np.float32), requires_grad=True)
    _, _, Dc = A.render_camera(scene, s["cam"], pos, rot, with_depth=True)
    assert torch.equal(Dc, Dd)
    (Dc * g_D).sum().backward()
    dc = rt.render_backward(torch.zeros((W, H, 3), device=dev), dL_dD=g_D, camera=True)
    assert torch.equal(pos.grad, dc["camera_position"].cpu()) and torch.equal(rot.grad, dc["camera_rotation"].cpu())
    # rays on the stored scene: no synchronisation, no rebuild
    sr = _scene_of("sh_depth16")
    rays_np = _ray_set(sr, n=1024, seed=4)
    R = rays_np.shape[0]
    gd = torch.randn(R, device=sr["dev"])
    direct = sr["scene"].render_rays_backward(_dev(rays_np, sr), torch.zeros((R, 3), device=sr["dev"]),
                                              rays_grad=True, dL_dD=gd)

    def refuse(*a, **k):
        raise AssertionError("render_rays updated or rebuilt the scene")

    lib = _native.load()
    rays = _dev(rays_np, sr).requires_grad_(True)
    torch.cuda.synchronize()
    with monkeypatch.context() as m:
        m.setattr(Scene, "set_gaussians", refuse)
        m.setattr(lib, "rtgs_scene_build_bvh", refuse)
        torch.cuda.set_sync_debug_mode("error")
        try:
            rgb_r, T_r, D_r = A.render_rays(sr["scene"], rays, with_depth=True)
            (D_r * gd).sum().backward()
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.equal(rays.grad, direct["rays"])


def test_depth_only_loss_on_ray_batches_recovers_positions_displaced_along_the_view_axis():
    import torch
    import rtgs.autograd as A
    from rtgs import _native
    torch.manual_seed(0)
    gs = random_set(400, seed=99, mean_scale=0.06)
    gs.opacity[:] = np.maximum(gs.opacity, 0.5)
    scene = make_scene(gs)
    dev = torch.device("cuda", scene.device)
    st = torch.cuda.current_stream(dev).cuda_stream
    fields, axes = [], []
    for th in np.linspace(0.0, 2 * np.pi, 4, endpoint=False):
        cam, ocam = make_camera(th, 1.1, 2.6, 96, 72)
        f = torch.empty((96, 72, 8), device=dev)
        _native.check(_native.load().rtgs_generate_rays(cam.native(), scene.device, f.data_ptr(), st))
        fields.append(f.reshape(-1, 8))
        axes.append(-np.asarray(ocam.position, np.float64) / np.linalg.norm(ocam.position))
    fields = torch.stack(fields)
    with torch.no_grad():
        targets = torch.stack([scene.render_rays(f, with_depth=True)[2] for f in fields])
    rng = np.random.default_rng(5)
    pos0 = gs.pos + 0.05 * rng.choice([-1.0, 1.0], (len(gs.pos), 1)) * axes[0][None, :]   # along view 0's axis
    p = {k: torch.tensor(np.asarray(v, np.float32), device=dev) for k, v in
         dict(pos=pos0, rot=gs.rot, scale=gs.scale, color=gs.color, opacity=gs.opacity, sh=gs.sh).items()}
    p["pos"].requires_grad_(True)
    opt = torch.optim.Adam([p["pos"]], lr=2e-3)
    P = fields.shape[1]
    gen = torch.Generator(device=dev).manual_seed(1)

    def full_loss():
        with torch.no_grad():
            _, _, D = A.render_rays(scene, fields.reshape(-1, 8), *(p[k] for k in GROUPS), with_depth=True)
            return float(((D - targets.reshape(-1)) ** 2).mean())

    loss0 = full_loss()
    for _ in range(150):
        views = torch.randperm(4, device=dev, generator=gen)[:2]
        pix = torch.randint(0, P, (2, 4096), device=dev, generator=gen)
        rays = fields[views[:, None], pix].reshape(-1, 8)
        want = targets[views[:, None], pix].reshape(-1)
        _, _, D = A.render_rays(scene, rays, *(p[k] for k in GROUPS), with_depth=True)
        loss = ((D - want) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
    loss1 = full_loss()
    err0 = np.abs(pos0 - gs.pos).mean()
    err1 = np.abs(p["pos"].detach().cpu().numpy() - gs.pos).mean()
    print(f"depth loss over all 4 views {loss0:.3e} -> {loss1:.3e}; mean position error {err0:.3e} -> {err1:.3e}")
    assert loss1 * 5 <= loss0 and err1 < err0
