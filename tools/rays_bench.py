#!/usr/bin/env python
"""Time the arbitrary-ray path on one GPU (rtgs_render_rays, rtgs_render_rays_backward) on the view and configuration
of tools/backward_bench.py.

    python tools/rays_bench.py [--config 1m_deg3_1080p] [--depth 16] [--t-cut 1e-4] [--iters 20] [--warmup 3]

Legs, each timed with CUDA events around `iters` calls after `warmup` calls of the same shape:
  field      rtgs_render_rays on the view's (W,H,8) ray field in field order (coherent: neighbouring threads trace
             neighbouring pixels), next to rtgs_render of the same view;
  permuted   the same rays in a random order (every warp's rays scattered over the image);
  batch      a training batch: 2^18 rays at random pixels of 8 orbit views;
and the backward of each, Gaussian gradients only (ray-gradient pointer NULL) and with the ray gradients too.  The
card's name and power limit are read in the same run.  Prints one JSON line.
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "rt-gaussian-splat-renderer_b200"), str(ROOT / "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from backward_bench import card_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="1m_deg3_1080p")
    ap.add_argument("--depth", type=int, default=16)
    ap.add_argument("--t-cut", type=float, default=1e-4)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1 << 18)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rays_bench needs a CUDA device")
    from rtgs import _native
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
    f = focal_from_fov(H, FOV_DEG)
    lib = _native.load()
    stream = lambda: torch.cuda.current_stream(dev).cuda_stream  # noqa: E731

    def field_of(theta):
        pos, rot = orbit_pose(theta, np.pi / 2, ORBIT_R)
        cam = Camera(pos, rot, (W, H), (f, f), device=0)
        rays = torch.empty((W * H, 8), device=dev)
        _native.check(lib.rtgs_generate_rays(cam.native(), 0, rays.data_ptr(), stream()))
        return cam, rays

    cam, field = field_of(0.0)   # view 0 of the orbit, as in backward_bench
    rt = RayTracer((W, H), scene, cam, t_cut=args.t_cut)
    gen = torch.Generator(device=dev).manual_seed(0)
    permuted = field[torch.randperm(W * H, device=dev, generator=gen)].contiguous()
    views = [field_of(th)[1] for th in np.linspace(0.0, 2 * np.pi, 8, endpoint=False)]
    pick_v = torch.randint(0, 8, (args.batch,), device=dev, generator=gen)
    pick_p = torch.randint(0, W * H, (args.batch,), device=dev, generator=gen)
    batch = torch.stack(views)[pick_v, pick_p].contiguous()
    del views

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.iters

    params = {k: torch.zeros_like(torch.as_tensor(a[k]), device=dev)
              for k in ("pos", "rot", "scale", "color", "opacity", "sh") if a[k] is not None}
    res = {"config": args.config, "n": n, "resolution": [W, H], "depth": args.depth, "t_cut": args.t_cut,
           "iters": args.iters, "warmup": args.warmup}
    out_rgb = torch.empty((W, H, 3), device=dev)
    out_T = torch.empty((W, H), device=dev)
    res["render_ms"] = round(timed(lambda: rt.render_device(args.depth, out=out_rgb, out_T=out_T)), 3)
    legs = {}
    for name, rays in (("field", field), ("permuted", permuted), ("batch", batch)):
        m = rays.shape[0]
        rgb = torch.empty((m, 3), device=dev)
        T = torch.empty(m, device=dev)
        d_rgb = torch.randn((m, 3), device=dev, generator=gen) * 1e-3
        d_T = torch.randn(m, device=dev, generator=gen) * 1e-3
        g_rays = torch.zeros((m, 8), device=dev)
        fwd = timed(lambda: _native.check(lib.rtgs_render_rays(scene.handle, m, rays.data_ptr(), args.depth,
                                                               args.t_cut, rgb.data_ptr(), T.data_ptr(), stream())))
        gptr = [params[k].data_ptr() if k in params else None for k in ("pos", "rot", "scale", "color", "opacity",
                                                                          "sh")]

        def bwd(gr):
            _native.check(lib.rtgs_render_rays_backward(scene.handle, m, rays.data_ptr(), args.depth, args.t_cut,
                                                        d_rgb.data_ptr(), d_T.data_ptr(), *gptr, gr, None, None,
                                                        stream()))

        legs[name] = {"rays": m, "forward_ms": round(fwd, 3),
                      "backward_gaussians_ms": round(timed(lambda: bwd(None)), 3),
                      "backward_with_ray_grads_ms": round(timed(lambda: bwd(g_rays.data_ptr())), 3)}
        legs[name]["forward_ns_per_ray"] = round(fwd * 1e6 / m, 2)
    # the coherent field against the frame render (the records hold float32-rounded directions)
    _native.check(lib.rtgs_render_rays(scene.handle, W * H, field.data_ptr(), args.depth, args.t_cut,
                                       out_rgb.data_ptr(), out_T.data_ptr(), stream()))
    ref = rt.render_device(args.depth)
    torch.cuda.synchronize()
    res["field_vs_render_max_abs"] = float((out_rgb - ref).abs().max())
    res["legs"] = legs
    res["card"] = card_info(torch)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
