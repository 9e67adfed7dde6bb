"""The precise hit test in the camera's pixel basis (render_common.cuh: stage_candidate / precise_test): the staged
record holds G0 = W D0, Gx = W Rx, Gy = W Ry, e0 and u_c, and a ray's entry distance is t1 = L u_c + L sigma.  These
scenes are where that form is most exposed - the cancellation of t1 near the camera (`near_t`), the band of the
sqrt(3)-sigma surface for needles and pancakes seen edge-on (`near_q`), the largest and smallest pixel offsets and L
(fov 170 and 1 degrees) and a camera quaternion that is not unit (|d| != 1).  Every route against the float64 oracle,
and the routes against each other: the frame kernel and the two launches bit for bit, the depth-slab lists and the
fused kernel bit for bit, the fused kernel and the lists within 1e-5."""
import numpy as np
import pytest

from oracle import ref_numpy as O

from gpu_util import compare, make_camera, make_scene, random_set

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _camera(pos, rot, W, H, fov):
    from rtgs.camera import Camera
    from rtgs.orbit import focal_from_fov
    f = focal_from_fov(H, fov)
    return Camera(pos, rot, (W, H), (f, f)), O.CameraParams(np.asarray(pos), np.asarray(rot), W, H, (f, f))


def _check_routes(gs, cam, ocam, depth=16):
    from rtgs.ray_tracer import RayTracer
    scene = make_scene(gs)
    ref = O.render(gs, ocam, depth=depth)["rgb"]
    rt = RayTracer(cam.buf_size, scene, cam, t_cut=0.0)
    imgs = {}
    for mode in (0, 2, 1):
        scene.set_option("render_mode", mode)
        imgs[mode] = rt.render(depth).copy()
        mx, ps, bad = compare(imgs[mode], ref, TOL)
        assert mx <= TOL, (mode, mx, ps, bad)
    assert np.array_equal(imgs[0], imgs[2])            # k_frame == k_tile_lists + k_shade_tiles
    assert np.abs(imgs[0] - imgs[1]).max() <= 1e-5     # k_render against the lists
    # every group through the depth-slab lists: the same pixels as with the fused kernel, bit for bit
    scene.set_option("render_mode", 0)
    scene.set_option("heavy_limit", 24)
    scene.set_option("heavy_lists", 0)
    forced = rt.render(depth).copy()
    scene.set_option("heavy_lists", 2)
    assert np.array_equal(rt.render(depth), forced)
    assert np.abs(forced - imgs[0]).max() <= 1e-5
    return ref


def test_camera_just_outside_large_ellipsoids():
    gs = random_set(2427, seed=11020, mean_scale=0.24913786492941115, sh=True)
    gs.pos[:, 2] *= 0.02
    cam, ocam = make_camera(2.52281928787616, 2.007240515427329, 0.25061865417331775, 96, 68, fov=31.5)
    ref = _check_routes(gs, cam, ocam)
    assert np.abs(ref).max() > 0.1


@pytest.mark.parametrize("shape", ["needles", "pancakes"])
def test_thin_gaussians_edge_on(shape):
    """Axis-aligned needles (one long axis) and pancakes (one short axis, normal along z), the camera in the plane
    z = 0: every pancake and the needles along x and y are seen edge-on, q of most rays lies near the band."""
    rng = np.random.default_rng(7 if shape == "needles" else 8)
    n = 1500
    pos = rng.uniform(-1, 1, (n, 3))
    pos[:, 2] *= 0.05
    long_, short = 0.15, 1.5e-3
    scale = np.full((n, 3), short)
    if shape == "needles":
        scale[np.arange(n), rng.integers(0, 3, n)] = long_
    else:
        scale[:, :2] = long_ * rng.uniform(0.5, 1.5, (n, 2))
    rot = np.tile([1.0, 0.0, 0.0, 0.0], (n, 1))
    gs = O.GaussianSet(pos=pos, rot=rot, scale=scale, color=rng.uniform(0, 1, (n, 3)),
                       opacity=rng.uniform(0.2, 0.99, n), sh=rng.normal(0, 0.15, (n, 15, 3)))
    cam, ocam = make_camera(0.6, np.pi / 2, 2.5, 120, 80, fov=40.0)
    ref = _check_routes(gs, cam, ocam)
    assert np.abs(ref).max() > 0.1


@pytest.mark.parametrize("fov", [170.0, 1.0])
def test_extreme_fields_of_view(fov):
    """fov 170: pixel offsets a, b up to 0.7 and L up to 16 across the image; fov 1: offsets of 1e-4 and L = 1."""
    gs = random_set(3000, seed=23, mean_scale=0.04 if fov > 100 else 0.004)
    from rtgs.orbit import orbit_pose
    pos, rot = orbit_pose(1.1, 1.3, 0.6 if fov > 100 else 2.5)
    cam, ocam = _camera(pos, rot, 97, 70, fov)
    ref = _check_routes(gs, cam, ocam)
    assert np.abs(ref).max() > 0.1


@pytest.mark.parametrize("qscale", [0.6, 1.7])
def test_non_unit_camera_quaternion(qscale):
    """The reference rotates the rays with the quaternion as given: |d| = |q|^2, so t1 = L (u_c + sigma) carries it."""
    from rtgs.orbit import orbit_pose
    gs = random_set(2500, seed=29, mean_scale=0.04)
    pos, rot = orbit_pose(2.2, 1.0, 2.3)
    cam, ocam = _camera(pos, np.asarray(rot, np.float64) * qscale, 88, 72, 55.0)
    ref = _check_routes(gs, cam, ocam)
    assert np.abs(ref).max() > 0.1
