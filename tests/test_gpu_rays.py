"""rtgs_render_rays / rtgs_render_rays_backward, Scene.render_rays(_backward) and rtgs.autograd.render_rays on the GPU:
the image and the gradients against the float64 reference for rays (tests/ref_rays.py), degenerate rays, identities
that need no oracle, agreement with the pixel paths (rtgs_render, rtgs_render_backward, rtgs_render_backward_camera),
determinism and accumulation, autograd, and a short optimisation on random ray batches of several views."""
import numpy as np
import pytest

from oracle import ref_numpy as O

import ref_grad_camera as RC
import ref_rays as RR
from gpu_util import make_camera, random_set
from test_gpu_backward import ATOMIC_TOL, CASES, GRAD_TOL, GROUPS, _rel

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-5
IDENTITY_TOL = 1e-5
CAMERA_CHAIN_TOL = 1e-4   # the ray records hold float32-rounded directions; the pixel kernel uses float64 ones


def _single():
    # one Gaussian: the root of its tree carries an empty child that points at leaf 0 again
    gs = O.GaussianSet(pos=[[0.1, -0.05, 0.0]], rot=[[0.1, 0.2, 0.0, 0.97]], scale=[[0.4, 0.25, 0.3]],
                       color=[[0.2, 0.7, 0.4]], opacity=[0.8], sh=np.full((1, 15, 3), 0.04))
    cam, ocam = make_camera(0.3, 1.2, 2.5, 40, 32, fov=50.0)
    return gs, cam, ocam, 16, 0.0, None


RAY_CASES = dict(CASES, single=_single)


def _scene_of(case):
    import torch
    from gpu_util import make_scene
    gs, cam, ocam, depth, t_cut, _ = RAY_CASES[case]()
    scene = make_scene(gs)
    return dict(gs=gs, cam=cam, ocam=ocam, depth=depth, t_cut=t_cut, scene=scene,
                dev=torch.device("cuda", scene.device))


def _random_rays(gs, n, seed, kinds=("origin", "inside", "scaled", "axis", "interval")):
    """Rays of several kinds: origins around the cloud aimed at it, origins inside Gaussians, directions scaled by
    0.1 ... 10, axis-parallel directions, random start / end intervals."""
    rng = np.random.default_rng(seed)
    pos = np.asarray(gs.pos, np.float64)
    lo, hi = pos.min(0), pos.max(0)
    rays = np.zeros((n, 8))
    o = rng.uniform(lo - 1.0, hi + 1.0, (n, 3))
    tgt = pos[rng.integers(0, len(pos), n)] + rng.normal(0, 0.05, (n, 3))
    k = np.arange(n) % len(kinds)
    inside = np.array([kinds[i] == "inside" for i in k])
    o[inside] = pos[rng.integers(0, len(pos), inside.sum())]
    d = tgt - o
    d[inside] = rng.normal(size=(inside.sum(), 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    scaled = np.array([kinds[i] == "scaled" for i in k])
    d[scaled] *= np.exp(rng.uniform(np.log(0.1), np.log(10.0), (scaled.sum(), 1)))
    axis = np.array([kinds[i] == "axis" for i in k])
    ax = rng.integers(0, 3, axis.sum())
    d[axis] = 0.0
    d[axis, ax] = rng.choice([-1.0, 1.0], axis.sum())
    d[axis] *= rng.uniform(0.5, 2.0, (axis.sum(), 1))
    o[axis] = tgt[axis] - 3.0 * d[axis]
    rays[:, :3], rays[:, 3:6] = o, d
    rays[:, 7] = np.inf
    itv = np.array([kinds[i] == "interval" for i in k])
    dist = np.linalg.norm(tgt - o, axis=1) / np.linalg.norm(d, axis=1)
    rays[itv, 6] = dist[itv] * rng.uniform(0.0, 0.9, itv.sum())
    rays[itv, 7] = dist[itv] * rng.uniform(1.0, 1.5, itv.sum())
    return rays.astype(np.float32)


def _ray_set(s, field=True, n=2048, seed=0):
    """float32 (R,8) rays: the camera's ray field followed by random rays."""
    parts = []
    if field:
        parts.append(RR.camera_ray_records(s["ocam"]).astype(np.float32))
    parts.append(_random_rays(s["gs"], n, seed))
    return np.concatenate(parts)


def _dev(x, s):
    import torch
    return torch.tensor(np.asarray(x), dtype=torch.float32, device=s["dev"])


@pytest.mark.parametrize("case", list(RAY_CASES))
def test_forward_parity_with_the_reference(case):
    import torch
    s = _scene_of(case)
    rays = _ray_set(s)
    rgb, T = s["scene"].render_rays(_dev(rays, s), depth=s["depth"], t_cut=s["t_cut"])
    torch.cuda.synchronize()
    ref = RR.render(s["gs"], rays.astype(np.float64), depth=s["depth"], t_cut=s["t_cut"])
    e_rgb = np.abs(rgb.cpu().numpy() - ref["rgb"].detach().numpy()).max()
    e_T = np.abs(T.cpu().numpy() - ref["T"].detach().numpy()).max()
    hit = (ref["nlayers"] > 0).mean()
    print(case, f"rgb {e_rgb:.1e} T {e_T:.1e} hit {hit:.2f}")
    assert hit > 0.05
    assert max(e_rgb, e_T) <= FWD_TOL


@pytest.mark.parametrize("case", ["axis", "sh_depth16", "nosh_depth4", "inside", "t_cut_1e-2", "single"])
def test_camera_field_renders_the_camera_image_and_the_backward_replays_it_bit_for_bit(case):
    import torch
    from rtgs import _native
    from rtgs.ray_tracer import RayTracer
    s = _scene_of(case)
    cam = s["cam"]
    W, H = cam.buf_size.x, cam.buf_size.y
    field = torch.empty((W, H, 8), dtype=torch.float32, device=s["dev"])
    _native.check(_native.load().rtgs_generate_rays(cam.native(), s["scene"].device, field.data_ptr(),
                                                    torch.cuda.current_stream(s["dev"]).cuda_stream))
    rgb, T = s["scene"].render_rays(field, depth=s["depth"], t_cut=s["t_cut"])
    assert tuple(rgb.shape) == (W, H, 3) and tuple(T.shape) == (W, H)
    rt = RayTracer(cam.buf_size, s["scene"], cam, t_cut=s["t_cut"])
    T2 = torch.empty((W, H), dtype=torch.float32, device=s["dev"])
    img = rt.render_device(s["depth"], out_T=T2)
    torch.cuda.synchronize()
    e = max((rgb - img).abs().max().item(), (T - T2).abs().max().item())
    print(case, f"against render_device {e:.1e}")
    assert e <= FWD_TOL
    g = torch.randn((W, H, 3), device=s["dev"])
    rep = s["scene"].render_rays_backward(field, g, depth=s["depth"], t_cut=s["t_cut"], replay=True, rays_grad=True)
    torch.cuda.synchronize()
    assert torch.equal(rep["rgb"], rgb) and torch.equal(rep["T"], T)


def test_degenerate_rays_and_no_rays():
    import torch
    s = _scene_of("sh_depth16")
    W, H = s["ocam"].width, s["ocam"].height
    mid = (W // 2) * H   # 64 rays of two columns in the middle of the view
    rays = RR.camera_ray_records(s["ocam"]).astype(np.float32)[mid:mid + 64].copy()
    bad = {1: (0, np.nan), 5: (4, np.inf), 9: (3, -np.inf), 17: (6, 5.0), 30: (7, np.nan)}
    for r, (c, v) in bad.items():
        rays[r, c] = v
    rays[17, 7] = 5.0        # start == end
    rays[22, 3:6] = 0.0      # d = 0
    bad_rows = sorted(list(bad) + [22])
    good = np.setdiff1d(np.arange(64), bad_rows)
    scene = s["scene"]
    d_rays = _dev(rays, s)
    rgb, T = scene.render_rays(d_rays, depth=16)
    clean, cleanT = scene.render_rays(_dev(rays[good], s), depth=16)
    g = torch.ones((64, 3), device=s["dev"])
    out = scene.render_rays_backward(d_rays, g, torch.ones(64, device=s["dev"]), depth=16, rays_grad=True)
    torch.cuda.synchronize()
    assert (rgb[bad_rows] == 0).all() and (T[bad_rows] == 1).all()
    assert (out["rays"][bad_rows] == 0).all()
    # neighbouring valid rays of the same warp are unaffected
    assert torch.equal(rgb[good], clean) and torch.equal(T[good], cleanT)
    assert (T[good] < 1).any()
    # no rays at all
    empty = torch.empty((0, 8), device=s["dev"])
    e_rgb, e_T = scene.render_rays(empty)
    e = scene.render_rays_backward(empty, torch.empty((0, 3), device=s["dev"]), rays_grad=True)
    torch.cuda.synchronize()
    assert e_rgb.shape == (0, 3) and e_T.shape == (0,) and e["rays"].shape == (0, 8)
    assert all(float(e[k].abs().sum()) == 0 for k in GROUPS)


@pytest.mark.parametrize("case", list(RAY_CASES))
def test_backward_parity_with_the_reference(case):
    import torch
    s = _scene_of(case)
    rays = _ray_set(s, n=1024, seed=1)
    R = rays.shape[0]
    rng = np.random.default_rng(5)
    g_rgb, g_T = rng.normal(size=(R, 3)), rng.normal(size=R)
    got = s["scene"].render_rays_backward(_dev(rays, s), _dev(g_rgb, s), _dev(g_T, s), depth=s["depth"],
                                          t_cut=s["t_cut"], rays_grad=True)
    torch.cuda.synchronize()
    ref = RR.grad(s["gs"], rays.astype(np.float64), g_rgb, g_T, depth=s["depth"], t_cut=s["t_cut"])
    errs = {}
    for k in GROUPS:
        if k == "sh" and s["gs"].sh is None:
            assert "sh" not in got
            continue
        assert np.linalg.norm(ref[k]) > 0, k
        errs[k] = _rel(got[k].cpu().numpy(), ref[k])
    gr = got["rays"].cpu().numpy()
    errs["o"] = _rel(gr[:, :3], ref["o"])
    errs["d"] = _rel(gr[:, 3:6], ref["d"])
    assert (gr[:, 6:] == 0).all()
    print(case, {k: f"{v:.1e}" for k, v in errs.items()})
    assert max(errs.values()) <= GRAD_TOL, errs


@pytest.mark.parametrize("case", ["sh_depth16", "nosh_depth16", "inside", "nonunit_quaternions"])
def test_identities_translation_and_direction_scale(case):
    import torch
    s = _scene_of(case)
    rays = _ray_set(s, n=2048, seed=2)
    R = rays.shape[0]
    rng = np.random.default_rng(6)
    got = s["scene"].render_rays_backward(_dev(rays, s), _dev(rng.normal(size=(R, 3)), s),
                                          _dev(rng.normal(size=R), s), depth=s["depth"], rays_grad=True)
    torch.cuda.synchronize()
    gr = got["rays"].cpu().numpy().astype(np.float64)
    so, gp = gr[:, :3].sum(0), got["pos"].cpu().numpy().astype(np.float64).sum(0)
    err_t = np.linalg.norm(so + gp) / np.linalg.norm(so)
    d = rays[:, 3:6].astype(np.float64)
    dot = np.abs((gr[:, 3:6] * d).sum(1)) / np.maximum(np.linalg.norm(gr[:, 3:6], axis=1) * np.linalg.norm(d, axis=1),
                                                        1e-30)
    print(case, f"translation {err_t:.1e}, max |dL/dd . d| / (|dL/dd| |d|) {dot.max():.1e}")
    assert err_t <= IDENTITY_TOL
    assert dot.max() <= IDENTITY_TOL


@pytest.mark.parametrize("case", ["axis", "sh_depth16", "nosh_depth16", "inside", "t_cut_1e-2"])
def test_camera_field_gradients_equal_the_pixel_backward(case):
    import torch
    from rtgs.ray_tracer import RayTracer
    from test_gpu_camera_grad import CAM
    s = _scene_of(case)
    cam = s["cam"]
    W, H = cam.buf_size.x, cam.buf_size.y
    rt = RayTracer(cam.buf_size, s["scene"], cam, t_cut=s["t_cut"])
    g = torch.randn((W, H, 3), device=s["dev"], generator=torch.Generator(device=s["dev"]).manual_seed(3))
    gT = torch.randn((W, H), device=s["dev"], generator=torch.Generator(device=s["dev"]).manual_seed(4))
    pix = rt.render_backward(g, gT, depth=s["depth"], camera=True)
    # the float32 ray field of the camera, as torch float64 leaves of the camera model
    leaves = [torch.tensor(np.asarray(v, np.float64), requires_grad=True)
              for v in (cam.position, cam.rotation, cam.focal_length)]
    o, d = RC.camera_rays(s["ocam"], *leaves)
    field = torch.zeros((W * H, 8), dtype=torch.float64)
    field[:, :3], field[:, 3:6], field[:, 7] = o.detach(), d.detach(), float("inf")
    field = field.to(torch.float32).to(s["dev"])
    out = s["scene"].render_rays_backward(field, g.reshape(-1, 3), gT.reshape(-1), depth=s["depth"],
                                          t_cut=s["t_cut"], rays_grad=True)
    torch.cuda.synchronize()
    errs = {k: _rel(out[k].cpu().numpy(), pix[k].cpu().numpy()) for k in GROUPS if k in pix}
    gr = out["rays"].cpu().to(torch.float64)
    chained = torch.autograd.grad([o.expand_as(d), d], leaves, [gr[:, :3], gr[:, 3:6]])
    cam_err = {k: _rel(c.numpy(), pix[k].cpu().numpy()) for k, c in zip(CAM, chained)}
    print(case, {k: f"{v:.1e}" for k, v in {**errs, **cam_err}.items()})
    assert max(errs.values()) <= GRAD_TOL, errs
    assert max(cam_err.values()) <= CAMERA_CHAIN_TOL, cam_err


def test_three_cameras_in_one_batch_sum_three_pixel_backwards():
    import torch
    from rtgs import _native
    from rtgs.ray_tracer import RayTracer
    from gpu_util import make_scene
    gs = random_set(800, seed=31, mean_scale=0.08)
    scene = make_scene(gs)
    dev = torch.device("cuda", scene.device)
    st = torch.cuda.current_stream(dev).cuda_stream
    fields, gs_rgb, gs_T = [], [], []
    ref = None
    for th, ph in ((0.4, 1.1), (1.9, 0.8), (3.5, 1.7)):
        cam, _ = make_camera(th, ph, 2.6, 48, 40)
        f = torch.empty((48, 40, 8), device=dev)
        _native.check(_native.load().rtgs_generate_rays(cam.native(), scene.device, f.data_ptr(), st))
        g = torch.randn((48, 40, 3), device=dev)
        gT = torch.randn((48, 40), device=dev)
        rt = RayTracer(cam.buf_size, scene, cam, t_cut=0.0)
        ref = rt.render_backward(g, gT, depth=16, grads=ref)
        fields.append(f.reshape(-1, 8))
        gs_rgb.append(g.reshape(-1, 3))
        gs_T.append(gT.reshape(-1))
    got = scene.render_rays_backward(torch.cat(fields), torch.cat(gs_rgb), torch.cat(gs_T), depth=16)
    torch.cuda.synchronize()
    for k in GROUPS:
        err = _rel(got[k].cpu().numpy(), ref[k].cpu().numpy())
        print(k, f"{err:.1e}")
        assert err <= ATOMIC_TOL, k


def test_ray_gradients_are_deterministic_and_accumulate_exactly():
    import torch
    s = _scene_of("sh_depth16")
    rays = _dev(_ray_set(s, n=4096, seed=3), s)
    R = rays.shape[0]
    g, gT = torch.randn((R, 3), device=s["dev"]), torch.randn(R, device=s["dev"])
    one = s["scene"].render_rays_backward(rays, g, gT, depth=16, rays_grad=True)["rays"]
    again = s["scene"].render_rays_backward(rays, g, gT, depth=16, rays_grad=True)["rays"]
    two = s["scene"].render_rays_backward(rays, g, gT, depth=16, rays_grad=True, grads={"rays": one.clone()})["rays"]
    torch.cuda.synchronize()
    assert one.abs().sum() > 0
    assert torch.equal(one, again)
    assert torch.equal(two, 2 * one)


def test_autograd_matches_the_direct_call_and_the_stored_scene_path_neither_syncs_nor_rebuilds(monkeypatch):
    import torch
    import rtgs.autograd as A
    from rtgs import _native
    from rtgs.scene import Scene
    s = _scene_of("sh_depth16")
    scene, dev = s["scene"], s["dev"]
    rays_np = _ray_set(s, n=1024, seed=4)
    R = rays_np.shape[0]
    g, gT = torch.randn((R, 3), device=dev), torch.randn(R, device=dev)
    direct = scene.render_rays_backward(_dev(rays_np, s), g, gT, depth=16, rays_grad=True)
    # with the Gaussian tensors: update + rebuild, gradients for them and for the rays
    gv = scene.read_gaussians()
    p = {k: torch.tensor(v, device=dev, requires_grad=True) for k, v in gv.items() if v is not None}
    rays = _dev(rays_np, s).requires_grad_(True)
    rgb, T = A.render_rays(scene, rays, p["pos"], p["rot"], p["scale"], p["color"], p["opacity"], p["sh"], depth=16)
    ((rgb * g).sum() + (T * gT).sum()).backward()
    for k in GROUPS:
        assert _rel(p[k].grad.cpu().numpy(), direct[k].cpu().numpy()) <= ATOMIC_TOL, k
    assert torch.equal(rays.grad, direct["rays"])
    # the stored scene: no update, no rebuild, no synchronisation, parameters untouched
    before = scene.read_gaussians()
    lb = {k: v.copy() for k, v in scene.read_lbvh().items()}

    def refuse(*a, **k):
        raise AssertionError("render_rays updated or rebuilt the scene")

    lib = _native.load()
    rays2 = _dev(rays_np, s).requires_grad_(True)
    torch.cuda.synchronize()
    with monkeypatch.context() as m:
        m.setattr(Scene, "set_gaussians", refuse)
        m.setattr(lib, "rtgs_scene_build_bvh", refuse)
        m.setattr(lib, "rtgs_scene_set_gaussians_device", refuse)
        torch.cuda.set_sync_debug_mode("error")
        try:
            rgb2, T2 = A.render_rays(scene, rays2, depth=16)
            ((rgb2 * g).sum() + (T2 * gT).sum()).backward()
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.equal(rgb2.detach(), rgb.detach())
    assert torch.equal(rays2.grad, direct["rays"])
    after = scene.read_gaussians()
    for k, v in before.items():
        assert (v is None and after[k] is None) or np.array_equal(v, after[k]), k
    scene._lbvh = None
    for k, v in scene.read_lbvh().items():
        assert np.array_equal(v, lb[k]), k
    with pytest.raises(ValueError):
        A.render_rays(scene, rays2, p["pos"], depth=16)   # some Gaussian tensors but not all


def test_optimisation_on_random_ray_batches_of_several_views():
    import torch
    import rtgs.autograd as A
    from rtgs import _native
    from gpu_util import make_scene
    torch.manual_seed(0)
    gs = random_set(2000, seed=4242, mean_scale=0.05)
    scene = make_scene(gs)
    dev = torch.device("cuda", scene.device)
    st = torch.cuda.current_stream(dev).cuda_stream
    fields = []
    for th in np.linspace(0.0, 2 * np.pi, 8, endpoint=False):
        cam, _ = make_camera(th, 1.1, 2.6, 128, 96)
        f = torch.empty((128, 96, 8), device=dev)
        _native.check(_native.load().rtgs_generate_rays(cam.native(), scene.device, f.data_ptr(), st))
        fields.append(f.reshape(-1, 8))
    fields = torch.stack(fields)                                     # (8, P, 8)
    with torch.no_grad():
        targets = torch.stack([scene.render_rays(f)[0] for f in fields])
    rng = np.random.default_rng(7)
    init = dict(pos=gs.pos + 0.2 * gs.scale.mean(1, keepdims=True) * rng.normal(size=gs.pos.shape),
                rot=gs.rot, scale=gs.scale,
                color=np.clip(gs.color + rng.normal(0, 0.15, gs.color.shape), 0.0, 1.0),
                opacity=np.clip(gs.opacity + rng.normal(0, 0.15, gs.opacity.shape), 0.05, 0.95),
                sh=gs.sh + rng.normal(0, 0.05, gs.sh.shape))
    p = {k: torch.tensor(np.asarray(v, np.float32), device=dev) for k, v in init.items()}
    for k in ("pos", "color", "opacity", "sh"):
        p[k].requires_grad_(True)
    opt = torch.optim.Adam([{"params": [p["pos"]], "lr": 2e-4}, {"params": [p["color"], p["sh"]], "lr": 1e-2},
                            {"params": [p["opacity"]], "lr": 1e-2}])
    P = fields.shape[1]
    gen = torch.Generator(device=dev).manual_seed(1)

    def full_loss():
        with torch.no_grad():
            rgb, _ = A.render_rays(scene, fields.reshape(-1, 8), *(p[k] for k in GROUPS))
            return float(((rgb - targets.reshape(-1, 3)) ** 2).mean())

    loss0 = full_loss()
    for _ in range(200):
        views = torch.randperm(8, device=dev, generator=gen)[:4]
        pix = torch.randint(0, P, (4, 4096), device=dev, generator=gen)
        rays = fields[views[:, None], pix].reshape(-1, 8)             # 16 k rays of 4 views
        want = targets[views[:, None], pix].reshape(-1, 3)
        rgb, _ = A.render_rays(scene, rays, *(p[k] for k in GROUPS))
        loss = ((rgb - want) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        with torch.no_grad():
            p["opacity"].clamp_(0.01, 0.99)
    loss1 = full_loss()
    print(f"loss over all 8 views {loss0:.3e} -> {loss1:.3e}")
    assert loss1 * 10 <= loss0
