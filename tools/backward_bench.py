#!/usr/bin/env python
"""Time the differentiable render path on one GPU: forward (rtgs_render), backward (rtgs_render_backward), the
backward with the camera gradient (rtgs_render_backward_camera, with every Gaussian gradient and camera only),
Scene.set_gaussians + LBVH rebuild, one whole rtgs.autograd step and one rtgs.autograd.render_camera step, on a
synthetic bench configuration.

    python tools/backward_bench.py [--config 1m_deg3_1080p] [--depth 16] [--t-cut 1e-4] [--iters 20] [--warmup 3]

Prints one JSON line.  Kernel times are CUDA events around `iters` launches after `warmup` launches of the same shape;
the update and the autograd step are host clocks around work that ends in a device synchronise (the rebuild
synchronises anyway).  Where the backward's time goes is split by running it three ways: dL = 0 (every pixel stops
after the traversal and the replayed forward), dL != 0 with every gradient pointer NULL (the back-to-front pass
without its atomics), and the full pass.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "rt-gaussian-splat-renderer_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "--id=" + str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:   # noqa: BLE001 - reported, not fatal
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="1m_deg3_1080p")
    ap.add_argument("--depth", type=int, default=16)
    ap.add_argument("--t-cut", type=float, default=1e-4)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("backward_bench needs a CUDA device")
    import rtgs.autograd as A
    from rtgs.camera import Camera
    from rtgs.orbit import focal_from_fov, orbit_pose
    from rtgs.ray_tracer import RayTracer
    from rtgs.scene import Scene
    from rtgs.synthetic import CONFIGS, FOV_DEG, ORBIT_R, make_scene

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    n, seed, deg, (W, H) = CONFIGS[args.config]
    a = make_scene(n, seed, deg)
    scene = Scene(device=0).from_arrays(a["pos"], a["rot"], a["scale"], a["color"], a["opacity"], a["sh"])
    pos, rot = orbit_pose(0.0, np.pi / 2, ORBIT_R)
    f = focal_from_fov(H, FOV_DEG)
    cam = Camera(pos, rot, (W, H), (f, f), device=0)
    rt = RayTracer((W, H), scene, cam, t_cut=args.t_cut)
    depth = args.depth
    gen = torch.Generator(device=dev).manual_seed(0)
    d_rgb = torch.randn((W, H, 3), device=dev, generator=gen) * 1e-3
    d_T = torch.randn((W, H), device=dev, generator=gen) * 1e-3
    zero_rgb = torch.zeros_like(d_rgb)
    params = {k: torch.tensor(a[k], device=dev) for k in ("pos", "rot", "scale", "color", "opacity", "sh")
              if a[k] is not None}
    grads = {k: torch.zeros_like(v) for k, v in params.items()}

    def timed(fn, iters=args.iters, warmup=args.warmup):
        for _ in range(warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def host_timed(fn, iters=args.iters, warmup=args.warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        t = []
        for _ in range(iters):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(t)), float(min(t))

    out_rgb = torch.empty((W, H, 3), device=dev)
    out_T = torch.empty((W, H), device=dev)
    fwd = timed(lambda: rt.render_device(depth, out=out_rgb, out_T=out_T))
    bwd = timed(lambda: rt.render_backward(d_rgb, d_T, depth=depth, grads=grads))
    bwd_replay_only = timed(lambda: rt.render_backward(zero_rgb, None, depth=depth, grads=grads))
    # every gradient pointer NULL: the C call directly (the wrapper always passes buffers)
    from rtgs import _native
    lib = _native.load()
    ncam = cam.native()
    stream = lambda: torch.cuda.current_stream(dev).cuda_stream  # noqa: E731
    bwd_no_atomics = timed(lambda: _native.check(lib.rtgs_render_backward(
        scene.handle, ncam, 0, 0, W, H, depth, args.t_cut, d_rgb.data_ptr(), d_T.data_ptr(),
        None, None, None, None, None, None, None, None, stream())))
    cam_grads = {k: torch.zeros(n, device=dev) for k, n in (("camera_position", 3), ("camera_rotation", 4),
                                                              ("camera_focal", 2))}
    bwd_cam = timed(lambda: rt.render_backward(d_rgb, d_T, depth=depth, grads={**grads, **cam_grads}, camera=True))
    bwd_cam_only = timed(lambda: _native.check(lib.rtgs_render_backward_camera(
        scene.handle, ncam, 0, 0, W, H, depth, args.t_cut, d_rgb.data_ptr(), d_T.data_ptr(),
        None, None, None, None, None, None, *(cam_grads[k].data_ptr() for k in cam_grads), None, None, stream())))
    upd_med, upd_min = host_timed(lambda: scene.set_gaussians(*(params[k] for k in params)), iters=max(5, args.iters // 2))
    build_ms = scene.build_ms

    p = {k: v.clone().requires_grad_(k in ("pos", "color", "opacity", "sh")) for k, v in params.items()}

    def step():
        rgb, T = A.render(scene, cam, p["pos"], p["rot"], p["scale"], p["color"], p["opacity"], p.get("sh"),
                          depth=depth, t_cut=args.t_cut)
        ((rgb * d_rgb).sum() + (T * d_T).sum()).backward()

    step_med, step_min = host_timed(step, iters=max(5, args.iters // 2))
    cpos = torch.tensor(np.asarray(cam.position, np.float32), device=dev, requires_grad=True)
    crot = torch.tensor(np.asarray(cam.rotation, np.float32), device=dev, requires_grad=True)

    def camera_step():
        rgb, T = A.render_camera(scene, cam, cpos, crot, depth=depth, t_cut=args.t_cut)
        ((rgb * d_rgb).sum() + (T * d_T).sum()).backward()

    cam_step_med, cam_step_min = host_timed(camera_step, iters=max(5, args.iters // 2))
    layers = None
    try:
        rt.render_device(depth, collect_stats=True)
        layers = rt.last_stats["layers"] / max(rt.last_stats["rays"], 1)
    except Exception:   # noqa: BLE001
        pass
    res = {
        "config": args.config, "n": n, "resolution": [W, H], "depth": depth, "t_cut": args.t_cut,
        "iters": args.iters, "warmup": args.warmup, "mean_layers_per_ray": layers,
        "forward_ms": round(fwd, 3),
        "backward_ms": round(bwd, 3),
        "backward_breakdown_ms": {
            "traversal_and_replay (dL = 0)": round(bwd_replay_only, 3),
            "plus back-to-front pass without atomics": round(bwd_no_atomics, 3),
            "plus atomics (full)": round(bwd, 3),
        },
        "backward_camera_ms": {"with every Gaussian gradient": round(bwd_cam, 3),
                               "camera only (Gaussian pointers NULL)": round(bwd_cam_only, 3)},
        "set_gaussians_and_rebuild_ms": {"median": round(upd_med, 3), "min": round(upd_min, 3),
                                         "build_device_ms": round(build_ms, 3)},
        "autograd_step_ms": {"median": round(step_med, 3), "min": round(step_min, 3)},
        "render_camera_step_ms": {"median": round(cam_step_med, 3), "min": round(cam_step_min, 3)},
        "card": card_info(torch),
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
