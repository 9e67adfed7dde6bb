"""rtgs_render_backward, Scene.set_gaussians and rtgs.autograd on the GPU: gradients against the float64 reference
gradient (oracle/ref_grad.py), the backward's replayed image against rtgs_render in every render mode, accumulation and
regions, no interference with later renders, and a short optimisation."""
import numpy as np
import pytest

from oracle import ref_grad as RG
from oracle import ref_numpy as O

from gpu_util import make_camera, random_set

pytestmark = pytest.mark.gpu

GROUPS = ("pos", "rot", "scale", "color", "opacity", "sh")
GRAD_TOL = 1e-5     # || g - g_ref || / || g_ref || per group (float32 atomics; observed <= 2.1e-6)
REPLAY_TOL = 1e-5
ATOMIC_TOL = 1e-5   # the same sums accumulated by float32 atomics in another order


def _axis():
    gs = O.GaussianSet(pos=[[0.0, 0.0, 0.0]], rot=[[0.0, 0.0, 0.0, 1.0]], scale=[[0.3, 0.2, 0.25]],
                       color=[[0.8, 0.3, 0.1]], opacity=[0.7], sh=np.full((1, 15, 3), 0.05))
    cam, ocam = make_camera(0.0, np.pi / 2, 3.0, 40, 32, fov=40.0)
    return gs, cam, ocam, 16, 0.0, None


def _config1():
    from rtgs.ply import read_ply
    from pathlib import Path
    a = O.activate(read_ply(Path(__file__).resolve().parent / "data" / "test.ply"), 30.0)
    cam, ocam = make_camera(0.0, np.pi / 2, 1.0, 256, 256, fov=90.0)
    return O.GaussianSet(**a), cam, ocam, 16, 0.0, None


def _random(sh, depth, seed, n=600, t_cut=0.0, tile=None, res=(64, 48), nonunit=False, opaque=False):
    gs = random_set(n, seed=seed, mean_scale=0.08, sh=sh)
    if nonunit:
        rng = np.random.default_rng(seed + 1)
        gs.rot[:] = (gs.rot * rng.uniform(0.6, 1.5, (n, 1))).astype(np.float32)
    if opaque:
        gs.opacity[:] = np.maximum(gs.opacity, 0.6)
    cam, ocam = make_camera(0.4, 1.1, 2.6, *res)
    return gs, cam, ocam, depth, t_cut, tile


def _inside():
    gs = random_set(1500, seed=77, mean_scale=0.08)
    cam, ocam = make_camera(2.0, 0.9, 0.3, 96, 72, fov=90.0)
    return gs, cam, ocam, 16, 0.0, None


def _ksat():
    from pathlib import Path
    g = np.load(Path(__file__).resolve().parent / "golden" / "reference_ksat_fp64.npz")
    gs = O.GaussianSet(g["pos"], g["rot"], g["scale"], g["color"], g["opacity"], g["sh"])
    res = int(g["res"])
    from rtgs.camera import Camera
    cam = Camera(g["cam_pos"], g["cam_rot"], (res, res), (float(g["focal"]),) * 2)
    ocam = O.CameraParams(g["cam_pos"], g["cam_rot"], res, res, (float(g["focal"]),) * 2)
    return gs, cam, ocam, 16, 0.0, None


CASES = {
    "axis": _axis,
    "config1": _config1,
    "sh_depth1": lambda: _random(True, 1, 11),
    "nosh_depth4": lambda: _random(False, 4, 12),
    "sh_depth16": lambda: _random(True, 16, 13),
    "nosh_depth16": lambda: _random(False, 16, 14),
    "sh_depth32": lambda: _random(True, 32, 15, n=1500),
    "ragged_tile": lambda: _random(True, 8, 16, n=800, res=(97, 61), tile=(13, 7, 45, 37)),
    "inside": _inside,
    "nonunit_quaternions": lambda: _random(True, 16, 17, nonunit=True),
    "ksat": _ksat,
    "t_cut_1e-2": lambda: _random(True, 16, 18, n=1500, t_cut=1e-2, opaque=True),
}


def _setup(case):
    import torch
    from rtgs.ray_tracer import RayTracer
    from gpu_util import make_scene
    gs, cam, ocam, depth, t_cut, tile = CASES[case]()
    scene = make_scene(gs)
    rt = RayTracer(cam.buf_size, scene, cam, t_cut=t_cut)
    W, H = cam.buf_size.x, cam.buf_size.y
    x0, y0, w, h = (0, 0, W, H) if tile is None else tile
    rng = np.random.default_rng(5)
    g_rgb = rng.normal(size=(w, h, 3))
    g_T = rng.normal(size=(w, h))
    dev = rt._dev
    return dict(gs=gs, cam=cam, ocam=ocam, depth=depth, t_cut=t_cut, tile=tile, scene=scene, rt=rt,
                region=(x0, y0, w, h), g_rgb=g_rgb, g_T=g_T,
                d_rgb=torch.tensor(g_rgb, dtype=torch.float32, device=dev),
                d_T=torch.tensor(g_T, dtype=torch.float32, device=dev))


def _ref(s):
    x0, y0, w, h = s["region"]
    ii, jj = np.meshgrid(np.arange(x0, x0 + w), np.arange(y0, y0 + h), indexing="ij")
    pixels = np.stack([ii.ravel(), jj.ravel()], -1)
    # ref_grad works in float64 from the float32 values the scene stores
    return RG.grad(s["gs"], s["ocam"], s["g_rgb"].reshape(-1, 3), s["g_T"].reshape(-1), depth=s["depth"],
                   t_cut=s["t_cut"], pixels=pixels)


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


@pytest.mark.parametrize("case", list(CASES))
def test_gradient_parity_with_the_reference(case):
    import torch
    s = _setup(case)
    got = s["rt"].render_backward(s["d_rgb"], s["d_T"], depth=s["depth"], tile=s["tile"], replay=True)
    torch.cuda.synchronize()
    ref = _ref(s)
    w, h = s["region"][2:]
    assert np.abs(got["rgb"].cpu().numpy() - ref["rgb"].reshape(w, h, 3)).max() <= REPLAY_TOL
    assert np.abs(got["T"].cpu().numpy() - ref["T"].reshape(w, h)).max() <= REPLAY_TOL
    errs = {}
    for k in GROUPS:
        if k == "sh" and s["gs"].sh is None:
            assert "sh" not in got
            continue
        errs[k] = _rel(got[k].cpu().numpy(), ref[k])
        assert np.linalg.norm(ref[k]) > 0, k
    print(case, {k: f"{v:.1e}" for k, v in errs.items()})
    assert max(errs.values()) <= GRAD_TOL, errs


@pytest.mark.parametrize("case", list(CASES))
def test_replay_equals_the_forward_in_every_render_mode(case):
    import torch
    s = _setup(case)
    rt, scene = s["rt"], s["scene"]
    rep = rt.render_backward(s["d_rgb"], s["d_T"], depth=s["depth"], tile=s["tile"], replay=True)
    x0, y0, w, h = s["region"]
    for mode in (0, 1, 2):
        scene.set_option("render_mode", mode)
        T = torch.empty((w, h), dtype=torch.float32, device=rt._dev)
        img = rt.render_device(s["depth"], tile=s["tile"], out_T=T)
        torch.cuda.synchronize()
        assert (img - rep["rgb"]).abs().max().item() <= REPLAY_TOL, mode
        assert (T - rep["T"]).abs().max().item() <= REPLAY_TOL, mode
    scene.set_option("render_mode", 0)


def test_two_calls_sum_and_regions_split_the_gradient():
    import torch
    s = _setup("sh_depth16")
    rt = s["rt"]
    one = rt.render_backward(s["d_rgb"], s["d_T"], depth=16)
    two = rt.render_backward(s["d_rgb"], s["d_T"], depth=16, grads={k: v.clone() for k, v in one.items()})
    for k in GROUPS:   # float32 atomics land in a different order each call: equal up to rounding
        assert _rel(two[k].cpu().numpy(), 2 * one[k].cpu().numpy()) <= ATOMIC_TOL, k
    # the gradient of a region == the full-image gradient with dL zero outside that region
    x0, y0, w, h = 9, 5, 30, 27
    mask = torch.zeros_like(s["d_T"])
    mask[x0:x0 + w, y0:y0 + h] = 1
    full = rt.render_backward(s["d_rgb"] * mask[..., None], s["d_T"] * mask, depth=16)
    part = rt.render_backward(s["d_rgb"][x0:x0 + w, y0:y0 + h].contiguous(), s["d_T"][x0:x0 + w, y0:y0 + h].contiguous(),
                              depth=16, tile=(x0, y0, w, h))
    for k in GROUPS:
        assert full[k].abs().sum() > 0
        assert _rel(part[k].cpu().numpy(), full[k].cpu().numpy()) <= ATOMIC_TOL, k


def test_backward_and_an_unchanged_update_leave_renders_bit_identical():
    import torch
    s = _setup("sh_depth16")
    rt, scene = s["rt"], s["scene"]
    for _ in range(2):   # the candidate-list pool settles to its size in the first frames
        rt.render_device(16)
    before = rt.render_device(16).clone()
    rt.render_backward(s["d_rgb"], s["d_T"], depth=16, replay=True)
    after = rt.render_device(16).clone()
    g = scene.read_gaussians()
    dev = rt._dev
    t = {k: torch.tensor(v, device=dev) for k, v in g.items() if v is not None}
    scene.set_gaussians(t["pos"], t["rot"], t["scale"], t["color"], t["opacity"], t["sh"])
    rebuilt = rt.render_device(16).clone()
    torch.cuda.synchronize()
    assert torch.equal(before, after) and torch.equal(before, rebuilt)


def test_set_gaussians_checks_and_state():
    import torch
    from rtgs import _native
    s = _setup("sh_depth16")
    scene, rt = s["scene"], s["rt"]
    g = scene.read_gaussians()
    dev = rt._dev
    t = {k: torch.tensor(v, device=dev) for k, v in g.items() if v is not None}
    with pytest.raises(ValueError):
        scene.set_gaussians(t["pos"], t["rot"], t["scale"], t["color"], t["opacity"])          # sh missing
    with pytest.raises(ValueError):
        scene.set_gaussians(t["pos"][:-1], t["rot"], t["scale"], t["color"], t["opacity"], t["sh"])
    with pytest.raises(ValueError):
        scene.set_gaussians(t["pos"].double(), t["rot"], t["scale"], t["color"], t["opacity"], t["sh"])
    # moved parameters: the scene renders what the oracle renders from them
    t["pos"] += 0.05
    t["color"] *= 0.5
    lib = _native.load()
    st = torch.cuda.current_stream(dev).cuda_stream
    _native.check(lib.rtgs_scene_set_gaussians_device(scene.handle, t["pos"].data_ptr(), t["rot"].data_ptr(),
                                                      t["scale"].data_ptr(), t["color"].data_ptr(),
                                                      t["opacity"].data_ptr(), t["sh"].data_ptr(), st))
    with pytest.raises(_native.RtgsError):   # no render before the rebuild
        rt.render_device(16)
    with pytest.raises(_native.RtgsError):
        rt.render_backward(s["d_rgb"], s["d_T"], depth=16)
    scene.set_gaussians(t["pos"], t["rot"], t["scale"], t["color"], t["opacity"], t["sh"])
    img = rt.render_device(16).cpu().numpy()
    gs = O.GaussianSet(**{k: v.cpu().numpy() for k, v in t.items()})
    ref = O.render(gs, s["ocam"], depth=16)["rgb"]
    assert np.abs(img - ref).max() <= 1e-3


def test_autograd_matches_render_device_and_the_direct_call():
    import torch
    import rtgs.autograd as A
    s = _setup("ragged_tile")
    rt, scene = s["rt"], s["scene"]
    for _ in range(2):   # the candidate-list pool settles to its size in the first frames
        rt.render_device(s["depth"], tile=s["tile"])
    g = scene.read_gaussians()
    dev = rt._dev
    p = {k: torch.tensor(v, device=dev, requires_grad=True) for k, v in g.items() if v is not None}
    rgb, T = A.render(scene, s["cam"], p["pos"], p["rot"], p["scale"], p["color"], p["opacity"], p["sh"],
                      depth=s["depth"], t_cut=s["t_cut"], tile=s["tile"])
    x0, y0, w, h = s["region"]
    T2 = torch.empty((w, h), dtype=torch.float32, device=dev)
    img = rt.render_device(s["depth"], tile=s["tile"], out_T=T2)
    assert torch.equal(rgb.detach(), img) and torch.equal(T.detach(), T2)
    ((rgb * s["d_rgb"]).sum() + (T * s["d_T"]).sum()).backward()
    direct = rt.render_backward(s["d_rgb"], s["d_T"], depth=s["depth"], tile=s["tile"])
    for k in GROUPS:
        assert _rel(p[k].grad.cpu().numpy(), direct[k].cpu().numpy()) <= ATOMIC_TOL, k


def test_optimisation_recovers_a_perturbed_scene():
    import torch
    import rtgs.autograd as A
    torch.manual_seed(0)
    gs = random_set(2000, seed=4242, mean_scale=0.05)
    from gpu_util import make_scene
    scene = make_scene(gs)
    cam, _ = make_camera(0.4, 1.1, 2.6, 128, 96)
    dev = torch.device("cuda", scene.device)
    tgt = {k: torch.tensor(getattr(gs, k), device=dev) for k in GROUPS}
    with torch.no_grad():
        target, _ = A.render(scene, cam, *(tgt[k] for k in GROUPS))
    rng = np.random.default_rng(7)
    init = dict(pos=gs.pos + 0.2 * gs.scale.mean(1, keepdims=True) * rng.normal(size=gs.pos.shape),
                rot=gs.rot, scale=gs.scale,
                color=np.clip(gs.color + rng.normal(0, 0.15, gs.color.shape), 0.0, 1.0),
                opacity=np.clip(gs.opacity + rng.normal(0, 0.15, gs.opacity.shape), 0.05, 0.95),
                sh=gs.sh + rng.normal(0, 0.05, gs.sh.shape))
    p = {k: torch.tensor(np.asarray(v, np.float32), device=dev) for k, v in init.items()}
    train = ("pos", "color", "opacity", "sh")
    for k in train:
        p[k].requires_grad_(True)
    opt = torch.optim.Adam([{"params": [p["pos"]], "lr": 2e-4}, {"params": [p["color"], p["sh"]], "lr": 1e-2},
                            {"params": [p["opacity"]], "lr": 1e-2}])
    losses = []
    for _ in range(200):
        rgb, _ = A.render(scene, cam, *(p[k] for k in GROUPS))
        loss = ((rgb - target) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        with torch.no_grad():
            p["opacity"].clamp_(0.01, 0.99)
        losses.append(loss.item())
    print(f"loss {losses[0]:.3e} -> {losses[-1]:.3e}")
    assert losses[-1] * 10 <= losses[0]
