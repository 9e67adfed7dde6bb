"""The float64 reference gradient (oracle/ref_grad.py) against the image oracle it restates, and the argument checks of
the backward / in-place update entry points (no GPU needed)."""
import copy
import ctypes

import numpy as np
import pytest

from oracle import ref_grad as RG
from oracle import ref_numpy as O


def _scene(n, seed, sh=True, unit=True):
    rng = np.random.default_rng(seed)
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    if not unit:
        q *= rng.uniform(0.7, 1.4, (n, 1))
    gs = O.GaussianSet(pos=rng.uniform(-0.5, 0.5, (n, 3)), rot=q, scale=np.exp(rng.normal(np.log(0.3), 0.3, (n, 3))),
                       color=rng.uniform(0.1, 0.9, (n, 3)), opacity=rng.uniform(0.2, 0.9, n),
                       sh=rng.normal(0, 0.2, (n, 15, 3)) if sh else None)
    return gs


def _camera(W=8, H=6):
    pos, rot = O.orbit_pose(0.4, np.pi / 2 - 0.2, 2.5)
    f = O.focal_from_fov(H, 50.0)
    return O.CameraParams(pos, rot, W, H, (f, f))


def _as_f64(gs):
    """A copy whose parameters are float64 arrays (GaussianSet stores float32; finite differences need float64)."""
    g = copy.deepcopy(gs)
    for k in RG.NAMES:
        v = getattr(g, k)
        if v is not None:
            setattr(g, k, np.asarray(v, np.float64).copy())
    return g


@pytest.mark.parametrize("sh", [True, False])
@pytest.mark.parametrize("depth", [1, 3, 16])
def test_forward_equals_ref_numpy(sh, depth):
    gs = _scene(12, seed=3 + depth, sh=sh, unit=False)
    cam = _camera(12, 10)
    want = O.render(gs, cam, depth=depth)
    got = RG.render(gs, cam, depth=depth)
    assert np.abs(got["rgb"].detach().numpy() - want["rgb"]).max() <= 1e-12
    assert np.abs(got["T"].detach().numpy() - want["T"]).max() <= 1e-12
    assert (want["nhit"] > 0).mean() > 0.5   # the view is not empty


def test_t_cut_stops_at_the_first_thin_layer():
    gs = _scene(12, seed=5, sh=False)
    gs.opacity[:] = 0.95
    cam = _camera(12, 10)
    full = RG.render(gs, cam, depth=16)
    cut = RG.render(gs, cam, depth=16, t_cut=1e-2)
    Tf, Tc = full["T"].detach().numpy(), cut["T"].detach().numpy()
    assert (Tc > Tf).any()              # some pixel stopped early
    assert (Tc[Tc > Tf] < 1e-2).all()   # and only below the threshold


@pytest.mark.parametrize("case", ["sh_unit", "nosh_nonunit", "sh_nonunit_depth2", "t_cut"])
def test_gradients_match_central_differences(case):
    sh = case.startswith("sh")
    unit = case == "sh_unit"
    depth = 2 if case.endswith("depth2") else 16
    t_cut = 0.05 if case == "t_cut" else 0.0
    gs = _as_f64(_scene(5, seed=11, sh=sh or case == "t_cut", unit=unit))
    if case == "t_cut":
        gs.opacity[:] = 0.9
    cam = _camera(8, 6)
    rng = np.random.default_rng(1)
    g_rgb = rng.normal(size=(cam.width, cam.height, 3))
    g_T = rng.normal(size=(cam.width, cam.height))
    ana = RG.grad(gs, cam, g_rgb, g_T, depth=depth, t_cut=t_cut)
    base = RG.render(gs, cam, depth=depth, t_cut=t_cut)
    if t_cut > 0:
        assert (base["T"].detach().numpy() < t_cut).any()   # the rule stops some pixel early

    def loss(g):
        out = RG.render(g, cam, depth=depth, t_cut=t_cut)
        assert np.array_equal(out["layers"]["idx"], base["layers"]["idx"]), "a perturbation changed a layer list"
        assert np.array_equal(out["nlayers"], base["nlayers"]), "a perturbation moved a t_cut stop"
        return float((out["rgb"].detach().numpy() * g_rgb).sum() + (out["T"].detach().numpy() * g_T).sum())

    for name in RG.NAMES:
        if getattr(gs, name) is None:
            continue
        val = getattr(gs, name)
        fd = np.zeros_like(val)
        for i in np.ndindex(val.shape):
            h = 1e-6 * max(1.0, abs(val[i]))
            gp, gm = copy.deepcopy(gs), copy.deepcopy(gs)
            getattr(gp, name)[i] += h
            getattr(gm, name)[i] -= h
            fd[i] = (loss(gp) - loss(gm)) / (2 * h)
        err = np.linalg.norm(ana[name] - fd) / max(np.linalg.norm(fd), 1e-30)
        assert np.linalg.norm(fd) > 0, name
        assert err <= 1e-6, (name, err)


def test_backward_entry_points_validate_without_a_gpu(lib):
    # argument validation happens before any CUDA call
    assert lib.rtgs_render_backward(None, None, 0, 0, 1, 1, 16, 0.0, None, None, None, None, None, None, None, None,
                                    None, None, None) == -1
    assert b"invalid argument" in lib.rtgs_last_error()
    assert lib.rtgs_scene_set_gaussians_device(None, None, None, None, None, None, None, None) == -1
    assert b"invalid argument" in lib.rtgs_last_error()
    from rtgs import _native
    cam = ctypes.pointer(_native.make_camera((0, 0, 3), (0, 0, 0, 1), (100, 100), 16, 16))
    # a NULL scene is refused before the camera, depth or t_cut are looked at
    assert lib.rtgs_render_backward(None, cam, 0, 0, 16, 16, 16, 0.0, None, None, None, None, None, None, None, None,
                                    None, None, None) == -1
