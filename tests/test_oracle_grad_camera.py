"""The float64 reference gradient with respect to the camera (tests/ref_grad_camera.py): the image against the
image oracle, the gradient against central finite differences with the layer lists held fixed, and the argument
checks of rtgs_render_backward_camera (no GPU needed)."""
import copy
import ctypes

import numpy as np
import pytest

from oracle import ref_numpy as O

import ref_grad_camera as RC
from test_oracle_grad import _as_f64, _camera, _scene


def _cam64(cam, position=None, rotation=None, focal=None):
    """A copy of ``cam`` holding float64 values (CameraParams rounds to float32 on construction; finite differences
    need float64)."""
    c = copy.copy(cam)
    c.position = np.asarray(cam.position if position is None else position, np.float64).copy()
    c.rotation = np.asarray(cam.rotation if rotation is None else rotation, np.float64).copy()
    f = [float(cam.focal[0]), float(cam.focal[1])] if focal is None else focal
    c.focal = (float(f[0]), float(f[1]))
    return c


@pytest.mark.parametrize("sh", [True, False])
@pytest.mark.parametrize("unit", [True, False])
def test_camera_leaf_image_equals_ref_numpy(sh, unit):
    gs = _scene(12, seed=21, sh=sh, unit=False)
    cam = _camera(12, 10)
    if not unit:
        cam = _cam64(cam, rotation=np.asarray(cam.rotation, np.float64) * 1.3)
    want = O.render(gs, cam, depth=16)
    got = RC.render(gs, cam, depth=16)
    assert all(got["params"][k].requires_grad for k in RC.CAM_NAMES)
    assert np.abs(got["rgb"].detach().numpy() - want["rgb"]).max() <= 1e-12
    assert np.abs(got["T"].detach().numpy() - want["T"]).max() <= 1e-12
    assert (want["nhit"] > 0).mean() > 0.5   # the view is not empty
    # the camera's own layer lists passed back in change nothing
    again = RC.render(gs, cam, depth=16, layers=got["layers"])
    assert np.array_equal(again["rgb"].detach().numpy(), got["rgb"].detach().numpy())


@pytest.mark.parametrize("case", ["sh_unit", "nosh_unit", "sh_nonunit", "nosh_nonunit", "t_cut"])
def test_camera_gradients_match_central_differences(case):
    sh = case.startswith("sh") or case == "t_cut"
    t_cut = 0.05 if case == "t_cut" else 0.0
    gs = _as_f64(_scene(5, seed=11, sh=sh, unit=case != "t_cut"))   # the t_cut scene of test_oracle_grad
    if case == "t_cut":
        gs.opacity[:] = 0.9
    cam = _cam64(_camera(8, 6))
    if case.endswith("nonunit"):
        cam.rotation = cam.rotation * 1.25
    rng = np.random.default_rng(2)
    g_rgb = rng.normal(size=(cam.width, cam.height, 3))
    g_T = rng.normal(size=(cam.width, cam.height))
    ana = RC.grad(gs, cam, g_rgb, g_T, depth=16, t_cut=t_cut)
    base = RC.render(gs, cam, depth=16, t_cut=t_cut)
    if t_cut > 0:
        assert (base["T"].detach().numpy() < t_cut).any()   # the rule stops some pixel early

    def loss(c):
        # the perturbed camera's own lists are the unperturbed camera's (asserted), and are passed in held fixed
        own = O.render(gs, c, depth=16, return_layers=True)["layers"]
        assert np.array_equal(own["idx"], base["layers"]["idx"]), "a perturbation changed a layer list"
        out = RC.render(gs, c, depth=16, t_cut=t_cut, layers=base["layers"])
        assert np.array_equal(out["nlayers"], base["nlayers"]), "a perturbation moved a t_cut stop"
        return float((out["rgb"].detach().numpy() * g_rgb).sum() + (out["T"].detach().numpy() * g_T).sum())

    vals = dict(cam_position=cam.position, cam_rotation=cam.rotation, cam_focal=np.asarray(cam.focal, np.float64))
    arg = dict(cam_position="position", cam_rotation="rotation", cam_focal="focal")
    for name in RC.CAM_NAMES:
        val = vals[name]
        fd = np.zeros_like(val)
        for i in range(val.size):
            h = 1e-6 * max(1.0, abs(val[i]))
            vp, vm = val.copy(), val.copy()
            vp[i] += h
            vm[i] -= h
            fd[i] = (loss(_cam64(cam, **{arg[name]: vp})) - loss(_cam64(cam, **{arg[name]: vm}))) / (2 * h)
        err = np.linalg.norm(ana[name] - fd) / max(np.linalg.norm(fd), 1e-30)
        assert np.linalg.norm(fd) > 0, name
        assert err <= 1e-6, (name, err)
    # scaling the quaternion scales every ray direction and changes no image: the gradient is orthogonal to q
    q = cam.rotation
    assert abs(ana["cam_rotation"] @ q) <= 1e-9 * np.linalg.norm(ana["cam_rotation"]) * np.linalg.norm(q)


def test_camera_backward_entry_point_validates_without_a_gpu(lib):
    # argument validation happens before any CUDA call
    assert lib.rtgs_render_backward_camera(None, None, 0, 0, 1, 1, 16, 0.0, *([None] * 14)) == -1
    assert b"invalid argument" in lib.rtgs_last_error()
    from rtgs import _native
    cam = ctypes.pointer(_native.make_camera((0, 0, 3), (0, 0, 0, 1), (100, 100), 16, 16))
    # a NULL scene is refused before the camera, depth or t_cut are looked at
    assert lib.rtgs_render_backward_camera(None, cam, 0, 0, 16, 16, 16, 0.0, *([None] * 14)) == -1
    assert b"invalid argument" in lib.rtgs_last_error()
