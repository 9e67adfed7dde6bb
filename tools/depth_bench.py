#!/usr/bin/env python
"""Time depth rendering against the same call without depth on one GPU, on the view and configuration of
tools/backward_bench.py and tools/rays_bench.py.

    python tools/depth_bench.py [--config 1m_deg3_1080p] [--depth 16] [--t-cut 1e-4] [--iters 20] [--warmup 3]
                                [--batch 262144] [--rounds 3]

Legs, each a pair (plain call, depth call) timed with CUDA events around `iters` calls after `warmup` calls of the
same shape, the two alternated over `rounds` rounds (the median is reported, and every round's values):
  frame_mode{0,1,2}   rtgs_render vs rtgs_render_depth of the whole frame in each render mode;
  shade_tiles         k_shade_tiles alone (mode 0), from the per-kernel event timing of RTGS_OPT_KERNEL_TIMING;
  backward            rtgs_render_backward_camera vs rtgs_render_backward_depth with dL_dD, every Gaussian and
                      camera gradient;
  rays / rays_backward  rtgs_render_rays(_depth) and rtgs_render_rays_backward(_depth) (ray gradients, dL_dD) on a
                      training batch of `batch` rays at random pixels of 8 orbit views.
The card's name and power limit are read in the same run.  Prints one JSON line.
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
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("depth_bench needs a CUDA device")
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

    cam, _ = field_of(0.0)
    rt = RayTracer((W, H), scene, cam, t_cut=args.t_cut)
    ncam = cam.native()
    depth, t_cut = args.depth, args.t_cut

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

    def pair(plain, with_depth, timer=timed):
        runs = [(timer(plain), timer(with_depth)) for _ in range(args.rounds)]
        p, d = float(np.median([r[0] for r in runs])), float(np.median([r[1] for r in runs]))
        return {"plain_ms": round(p, 4), "depth_ms": round(d, 4), "ratio": round(d / p, 4),
                "rounds": [[round(x, 4), round(y, 4)] for x, y in runs]}

    out_rgb = torch.empty((W, H, 3), device=dev)
    out_T = torch.empty((W, H), device=dev)
    out_D = torch.empty((W, H), device=dev)
    res = {"config": args.config, "n": n, "resolution": [W, H], "depth": depth, "t_cut": t_cut,
           "iters": args.iters, "warmup": args.warmup, "rounds": args.rounds}
    for mode in (0, 1, 2):
        scene.set_option("render_mode", mode)
        res[f"frame_mode{mode}"] = pair(lambda: rt.render_device(depth, out=out_rgb, out_T=out_T),
                                        lambda: rt.render_device(depth, out=out_rgb, out_T=out_T, out_depth=out_D))
    scene.set_option("render_mode", 0)

    # k_shade_tiles alone: the second of the frame's three event-bracketed launches
    def shade_timer(fn):
        for _ in range(args.warmup):
            fn()
        scene.set_option("kernel_timing", args.iters)
        for _ in range(args.iters):
            fn()
        ms = scene.read_kernel_times(args.iters)
        scene.set_option("kernel_timing", 0)
        return float(np.mean(ms[:, 1]))

    res["shade_tiles"] = pair(lambda: rt.render_device(depth, out=out_rgb, out_T=out_T),
                              lambda: rt.render_device(depth, out=out_rgb, out_T=out_T, out_depth=out_D), shade_timer)

    gen = torch.Generator(device=dev).manual_seed(0)
    d_rgb = torch.randn((W, H, 3), device=dev, generator=gen) * 1e-3
    d_T = torch.randn((W, H), device=dev, generator=gen) * 1e-3
    d_D = torch.randn((W, H), device=dev, generator=gen) * 1e-3
    grads = [torch.zeros((n,) + s, device=dev) for s in ((3,), (4,), (3,), (3,), (), (15, 3))]
    if a["sh"] is None:
        grads[5] = None
    cgr = [torch.zeros(k, device=dev) for k in (3, 4, 2)]
    ptrs = [None if g is None else g.data_ptr() for g in grads] + [g.data_ptr() for g in cgr]
    head = lambda: (scene.handle, ncam, 0, 0, W, H, depth, t_cut, d_rgb.data_ptr(), d_T.data_ptr(), *ptrs)  # noqa: E731
    res["backward"] = pair(
        lambda: _native.check(lib.rtgs_render_backward_camera(*head(), None, None, stream())),
        lambda: _native.check(lib.rtgs_render_backward_depth(*head(), None, None, d_D.data_ptr(), None, stream())))

    views = [field_of(th)[1] for th in np.linspace(0.0, 2 * np.pi, 8, endpoint=False)]
    pick_v = torch.randint(0, 8, (args.batch,), device=dev, generator=gen)
    pick_p = torch.randint(0, W * H, (args.batch,), device=dev, generator=gen)
    batch = torch.stack(views)[pick_v, pick_p].contiguous()
    del views
    m = batch.shape[0]
    r_rgb, r_T, r_D = (torch.empty((m, 3), device=dev), torch.empty(m, device=dev), torch.empty(m, device=dev))
    g_rgb = torch.randn((m, 3), device=dev, generator=gen) * 1e-3
    g_T = torch.randn(m, device=dev, generator=gen) * 1e-3
    g_D = torch.randn(m, device=dev, generator=gen) * 1e-3
    g_rays = torch.zeros((m, 8), device=dev)
    rhead = (scene.handle, m, batch.data_ptr(), depth, t_cut)
    res["rays"] = pair(
        lambda: _native.check(lib.rtgs_render_rays(*rhead, r_rgb.data_ptr(), r_T.data_ptr(), stream())),
        lambda: _native.check(lib.rtgs_render_rays_depth(*rhead, r_rgb.data_ptr(), r_T.data_ptr(), r_D.data_ptr(),
                                                         stream())))
    bargs = (*rhead, g_rgb.data_ptr(), g_T.data_ptr(), *ptrs[:6], g_rays.data_ptr(), None, None)
    res["rays_backward"] = pair(
        lambda: _native.check(lib.rtgs_render_rays_backward(*bargs, stream())),
        lambda: _native.check(lib.rtgs_render_rays_backward_depth(*bargs, g_D.data_ptr(), None, stream())))
    res["batch"] = m
    res["card"] = card_info(torch)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
