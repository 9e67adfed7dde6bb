#!/usr/bin/env python
"""bench.py — Mrays/s of the per-ray render path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]

Workload (config 3 of BASELINE.json, the one the metric is quoted on): synthetic 1 M random
Gaussians, SH degree 3, seed 1002, 1920x1080, vertical fov 60 deg, orbit radius 2.2, depth 16.
A "step" = ONE full 1080p frame (ray generation + LBVH traversal + intersection + 16-nearest
k-buffer + SH compositing + framebuffer write) of one view of the 64-view orbit (config 5); the
step s on rank r renders view (s*N + r) mod 64, view 0 being config 3's camera.  One ray = one finished pixel.

Multi-GPU (one process per GPU, scene replicated, NO collective on the data path):
  views  (value, e2e; "scaling": "weak")  rank r renders its views; at N > 1 every rank's kernels store their frame
         straight into GPU 0's memory over NVLink (rtgs.sharding.PeerFrame) and GPU 0 waits for the device-side
         arrival counters, so a step ends with all N frames resident on GPU 0 (SURVEY.md 8d)
  tiles  ("tiles": BASELINE config 3; "tiles_config4": config 4 at 8 GPUs) every frame is cut into 32-column stripes
         dealt round-robin; strong scaling of one frame, speed-up against rank 0 rendering the whole frame alone in
         the same process, bit-identity checked, slowest kernel named per rank

value  = whole-job Mrays/s with everything resident in HBM: K steps alternating on two CUDA streams (two frames in
         flight per GPU, the way the sweep API runs), CUDA events around both, max over ranks;
         serial_value = the same K steps on one stream (this loop also carries the per-kernel events)
e2e    = the same through the public API with HOST buffers: the orbit sweep as a user writes it with
         RayTracer.render_async()/result() (camera struct in, image delivered to pinned host memory, every step,
         inside the timed region; two frames in flight) or the blocking RayTracer.render() loop, whichever is faster
         (both reported); e2e.compact = the opt-in 8-bit delivery
roofline = the dominant kernel, k_shade_tiles (intersection + k-buffer + SH compositing): algorithmic bytes per
         ray (SURVEY.md §8d: 16 + kbar*(64 + 192[sh]), all of them consumed by this kernel) x rays per launch /
         its mean duration, measured with CUDA events the library records around each kernel on the render
         stream during the serial timed loop, against the measured HBM copy bandwidth in MEASURED_PEAKS.json;
         "kernels" lists every kernel of the step with its mean time and share
cpu_baseline = oracle/ref_cpu.cpp (reference-shaped C++/OpenMP port, float32, every core this process may use)
         on a pixel subsample

Steps: value, serial_value and e2e run exactly K timed steps.  To bound the run time, the secondary legs cap K
and report what they ran: tiles min(K, 128) frames and tiles_config4 min(K, 32) ("frames"), cpu_baseline
min(K, 32) steps ("steps"; --impl reference runs K).

--dump-outputs DIR writes the frame of the last timed step of the one-stream (serial_value) loop as DIR/frame.npy
((W,H,3) float32; at N > 1 every rank's frame, DIR/frame_rank<r>.npy, written by rank 0), read back untimed.  It is
not taken from the two-stream loop that gives `value`: there both streams store into one buffer, so what that loop
leaves behind need not be a single step's frame; both loops render the same views.  The inputs are seeded, so two
builds run with the same arguments compare output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "rt-gaussian-splat-renderer_b200"))

N_VIEWS = 64
DEPTH = 16
T_CUT = 1e-4
FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback
DUMP_MAX_BYTES = 64_000_000


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="1m_deg3_1080p")
    ap.add_argument("--no-tiles", action="store_true",
                    help="skip the tile-sharded (strong-scaling) measurement that follows the view-sharded one")
    ap.add_argument("--tile-modes", default="0,2",
                    help="render modes tried for the tile-sharded frames (0 = two launches, 2 = one-launch frame kernel); "
                         "the faster one is reported, all are listed")
    ap.add_argument("--config4", action="store_true",
                    help="also measure BASELINE config 4 (3 M Gaussians, 3840x2160, tiles over all GPUs); default at 8 GPUs")
    ap.add_argument("--h-target", type=float, default=None,
                    help="diagnostic: expected ellipsoid crossings per cube-spanning ray of the synthetic scene "
                         "(default 16, SURVEY.md 8d); larger = bigger Gaussians, denser tiles")
    ap.add_argument("--morton-bits", type=int, default=0, choices=[0, 30, 63],
                    help="LBVH code width: 0 = automatic (30, the north-star spec, unless the codes are degenerate), "
                         "30, 63 (the wide variant for scenes with outliers)")
    ap.add_argument("--outliers", type=int, default=0,
                    help="diagnostic: move this many Gaussians ~4000 scene radii away (what stray points of a "
                         "trained scene do to 10-bit-per-axis Morton codes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-stride", type=int, default=0, help="pixel subsample stride of the CPU legs (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step (one-stream loop) as DIR/frame.npy, (W,H,3) float32; "
                         "at N > 1, rank 0 writes every rank's frame as DIR/frame_rank<r>.npy.  Above 64 MB in all, "
                         "every file keeps the same fixed, seeded sample of pixels, as (n,3)")
    return ap.parse_args()


def make_views(W, H, n_views=N_VIEWS, phi=np.pi / 2):
    from rtgs.orbit import focal_from_fov, orbit_pose
    from rtgs.synthetic import FOV_DEG, ORBIT_R
    f = focal_from_fov(H, FOV_DEG)
    return f, [orbit_pose(2 * np.pi * k / n_views, phi, ORBIT_R) for k in range(n_views)]


def load_config(name, h_target=None):
    """(arrays, n, seed, sh_degree, (W, H), n_views, phi, description) of a bench configuration."""
    from rtgs.synthetic import CONFIGS, SURFACE_CONFIGS, make_scene, make_surface_scene
    if name in SURFACE_CONFIGS:
        n, seed, res, nv, phi = SURFACE_CONFIGS[name]
        return (make_surface_scene(n, seed), n, seed, 3, res, nv, phi,
                f"synthetic {n} Gaussians on surfaces (6 shells + a floor, flat splats, log-normal sizes sigma 1, 40 huge "
                f"translucent blobs, 6 stray points 800 radii out), SH degree 3, seed {seed}")
    n, seed, deg, res = CONFIGS[name]
    arrays = make_scene(n, seed, deg) if h_target is None else make_scene(n, seed, deg, h_target)
    return arrays, n, seed, deg, res, N_VIEWS, np.pi / 2, f"synthetic {n} random Gaussians, SH degree {deg}, seed {seed}"


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every few ms DURING the timed region
    (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints)."""

    def __init__(self, index, period_s=0.002):
        self.index, self.period, self.samples, self.reasons = index, period_s, [], set()
        self.stop_flag = threading.Event()
        self.thread = None
        self.max_mhz = None
        self.power_w = []

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
                if len(self.samples) % 8 == 1:   # the power query can take tens of milliseconds
                    self.power_w.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self.stop_flag.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "power_w_max": max(self.power_w) if self.power_w else None}


def load_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(kernel):
    """dram bytes per launch of `kernel` from the committed ncu summary (profiles/), if any."""
    p = ROOT / "profiles" / "render_kernel_traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text())[kernel]["dram_bytes_per_launch"]
        except Exception:
            return None
    return None


def cpu_leg(cfg_name, scene_arrays, W, H, focal, views, steps, warmup, stride):
    """The reference-shaped CPU port (float32, all host threads) on a pixel subsample."""
    from oracle import ref_cpu
    from oracle import ref_numpy as O
    ref_cpu.build()
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must use every core this process may run on
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    t0 = time.perf_counter()
    cs = ref_cpu.CpuScene(scene_arrays["pos"], scene_arrays["rot"], scene_arrays["scale"], scene_arrays["color"],
                          scene_arrays["opacity"], scene_arrays["sh"])
    build_s = time.perf_counter() - t0
    pix = ref_cpu.all_pixels(W, H, stride)
    times = []
    for s in range(warmup + steps):
        pos, rot = views[s % len(views)]
        cam = O.CameraParams(np.asarray(pos), np.asarray(rot), W, H, (focal, focal))
        t0 = time.perf_counter()
        cs.render(cam, DEPTH, pixels=pix, precision="float", threads=threads)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    total = sum(times)
    return {"mrays": pix.shape[0] * len(times) / total / 1e6, "ms_per_step": 1e3 * total / len(times),
            "cores": threads, "rays_per_step": int(pix.shape[0]), "build_s": build_s, "steps": len(times),
            "sample": f"every {stride}th column and row of each {W}x{H} view ({pix.shape[0]} rays/step), "
                      f"{len(times)} steps, float32, K={DEPTH} closest-hit restarts over the LBVH"}


def dump_outputs(path, frames, max_bytes=DUMP_MAX_BYTES):
    """Write `frames` (name -> (W,H,3) float32 array) as path/<name>.npy, at most `max_bytes` in all: above that every
    file keeps the same seeded sample of pixels, so two runs with the same arguments compare pixel for pixel."""
    path = Path(path)
    path.mkdir(parents=True, exist_ok=True)
    header = 128                                        # bytes of the .npy header of an array of up to 3 dimensions
    W, H, _ = next(iter(frames.values())).shape
    npix = W * H
    total = sum(a.nbytes + header for a in frames.values())
    if total > max_bytes:
        keep = (max_bytes - header * len(frames)) * npix // (total - header * len(frames))
        idx = np.sort(np.random.default_rng(0).choice(npix, size=keep, replace=False))
        frames = {k: a.reshape(npix, -1)[idx] for k, a in frames.items()}
    for k, a in frames.items():
        np.save(path / f"{k}.npy", np.ascontiguousarray(a, dtype=np.float32))


def views_of(W, H):
    return make_views(W, H)


class TwoStreams:
    """Two CUDA streams used alternately, frame by frame, bracketed by events on the default stream: frames on
    different streams use different frame scratch in the library (csrc/render.cu), so the head of frame f+1
    overlaps the tail of frame f on the device."""

    def __init__(self, torch, n=2):
        self.torch = torch
        self.streams = [torch.cuda.Stream() for _ in range(n)]

    def begin(self):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        for s in self.streams:
            s.wait_event(e)
        return e

    def stream(self, k):
        return self.torch.cuda.stream(self.streams[k % len(self.streams)])

    def end(self):
        cur = self.torch.cuda.current_stream()
        for s in self.streams:
            cur.wait_stream(s)
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        return e


def allmax(dist, torch, vals):
    if dist is None:
        return list(vals)
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def allgather(dist, torch, vals, world):
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    if dist is None:
        return [t.tolist()]
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [o.tolist() for o in out]


def measure_tiles(torch, dist, rank, world, local_rank, scene, rt, cam, views, W, H, steps, warmup, barrier, modes):
    """Strong scaling of ONE frame (BASELINE configs 3 / 4): 32-pixel column stripes dealt round-robin to the ranks,
    every rank's kernels store straight into rank 0's framebuffer over NVLink (rtgs.sharding.PeerFrame), hand-over
    by device-side counters - no collective, no host synchronisation.  Measures, in the same processes:
      t1   rank 0 alone renders the whole frame (the 1-GPU reference of the speed-up), latency and two-stream
      tN   all ranks, one frame in flight per rank (frame latency) and frames alternating on two streams (throughput)
    and verifies the assembled frame bit for bit against rank 0's own full render."""
    from rtgs.sharding import PeerFrame
    res = {}
    out_local = torch.empty((W, H, 3), dtype=torch.float32, device="cuda")
    ts = TwoStreams(torch)
    nv = len(views)

    def set_view(s):
        cam.position, cam.rotation = views[s % nv]

    def timed(step_fn, two_streams, n_warm, n_steps):
        for s in range(n_warm):
            set_view(s)
            step_fn(s, None)
        barrier()
        if two_streams:
            e0 = ts.begin()
            for s in range(n_steps):
                set_view(s)
                with ts.stream(s):
                    step_fn(s, None)
            e1 = ts.end()
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(n_steps):
                set_view(s)
                step_fn(s, None)
            e1.record()
        barrier()
        return e0.elapsed_time(e1) / n_steps

    # ---- 1-GPU reference on rank 0 (whole frames, same views), in each candidate render mode
    scene.set_stripe()
    single = {}
    for mode in modes:
        scene.set_option("render_mode", mode)
        if rank == 0:
            single[mode] = (timed(lambda s, _: rt.render_device(DEPTH, out=out_local), False, warmup, steps),
                            timed(lambda s, _: rt.render_device(DEPTH, out=out_local), True, warmup, steps))
        else:
            barrier(); barrier(); barrier(); barrier()
    t1_lat = min(v[0] for v in single.values()) if rank == 0 else 0.0
    t1_pipe = min(min(v) for v in single.values()) if rank == 0 else 0.0

    # ---- all ranks: stripes into rank 0's frame
    peer = PeerFrame(W, H, rank, world, local_rank, dist, slots=1, buffers=4)
    scene.set_stripe(world, rank)

    local = [torch.empty((W, H, 3), dtype=torch.float32, device="cuda") for _ in range(2)]

    def tile_step(s, _):
        # gather by STORES: the render kernels write their stripes into rank 0's frame over NVLink as they go
        rt.render_device(DEPTH, out=peer.begin(scene))
        if rank == 0:
            peer.wait()
            peer.release()

    def tile_step_copy(s, _):
        # gather by COPY: render into local memory, then one strided copy of the rank's stripes over NVLink
        peer.begin_copy()
        rt.render_device(DEPTH, out=local[s % 2])
        peer.deliver_stripes(local[s % 2])
        if rank == 0:
            peer.wait()
            peer.release()

    per_mode = {}
    variants = [(m, "stores") for m in modes] + ([(modes[0], "copy")] if world > 1 else [])
    for mode, gather in variants:
        step = tile_step if gather == "stores" else tile_step_copy
        scene.set_option("render_mode", mode)
        lat = timed(step, False, warmup, steps)
        pipe = timed(step, True, warmup, steps)
        scene.set_option("kernel_timing", min(steps, 256))
        timed(step, False, 0, min(steps, 256))
        kt = scene.read_kernel_times(min(steps, 256)).astype(np.float64).mean(axis=0)
        scene.set_option("kernel_timing", 0)
        lat, pipe = allmax(dist, torch, [lat, pipe])
        per_rank = allgather(dist, torch, kt.tolist(), world)
        per_mode[(mode, gather)] = {"ms_per_frame": lat, "ms_per_frame_two_streams": pipe,
                                    "kernel_names": list(scene.kernel_names),
                                    "kernels_ms_per_rank": [[round(v, 5) for v in r] for r in per_rank]}
    best = min(per_mode, key=lambda m: min(per_mode[m]["ms_per_frame_two_streams"], per_mode[m]["ms_per_frame"]))
    scene.set_option("render_mode", best[0])
    best_step = tile_step if best[1] == "stores" else tile_step_copy

    # ---- untimed check: the assembled frame == rank 0's own full-frame render, bit for bit
    set_view(0)
    torch.cuda.synchronize()
    barrier()
    best_step(0, None)
    torch.cuda.synchronize()
    barrier()
    verified = None
    if rank == 0:
        assembled = peer.frame().clone()
        scene.set_stripe()
        set_view(0)
        full = rt.render_device(DEPTH, out=out_local)
        torch.cuda.synchronize()
        verified = bool(torch.equal(full, assembled))
        scene.set_stripe(world, rank)
    barrier()

    # ---- end to end: every frame delivered to HOST memory.  Each rank copies its own stripes into one shared,
    # page-locked host image over its own PCIe link (rtgs.sharding.HostFrame); rank 0's host thread collects every
    # frame inside the timed region.  Nothing is gathered on a device, no collective.
    from rtgs.sharding import HostFrame
    hf = HostFrame(W, H, rank, world, local_rank, dist, buffers=3)
    dev = [torch.empty((W, H, 3), dtype=torch.float32, device="cuda") for _ in range(2)]

    def e2e_loop(n):
        last = None
        for s in range(n):
            set_view(s)
            with ts.stream(s):
                rt.render_device(DEPTH, out=dev[s % 2])
                hf.deliver(dev[s % 2])
            if rank == 0 and s >= 1:
                last = hf.wait()
                hf.release()
        if rank == 0:
            last = hf.wait()
            hf.release()
        return last

    e2e_loop(3)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    e2e_loop(steps)
    torch.cuda.synchronize()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / steps
    (e2e_ms,) = allmax(dist, torch, [e2e_ms])
    # untimed check of the host path: one frame through it == rank 0's own full render
    host_verified = None
    set_view(0)
    rt.render_device(DEPTH, out=dev[0])
    hf.deliver(dev[0])
    if rank == 0:
        got = np.array(hf.wait(), copy=True)
        hf.release()
        scene.set_stripe()
        set_view(0)
        full = rt.render_device(DEPTH, out=out_local)
        torch.cuda.synchronize()
        host_verified = bool(np.array_equal(full.cpu().numpy(), got))
        scene.set_stripe(world, rank)
    torch.cuda.synchronize()
    barrier()
    hf.close()
    scene.set_stripe()
    scene.set_option("render_mode", modes[0])
    peer.close()
    if rank != 0:
        return None
    b = per_mode[best]
    k = b["kernels_ms_per_rank"]
    kmax = [max(r[i] for r in k) for i in range(3)]
    dom = int(np.argmax(kmax))
    tput = min(b["ms_per_frame_two_streams"], b["ms_per_frame"])     # frames per second of a sweep: the better schedule
    res = {"resolution": [W, H], "frames": steps, "render_mode": best[0],
           "gather": ("peer stores from the render kernels" if best[1] == "stores" else
                      "render into local memory + one strided peer copy of the rank's stripes") +
                     " + device-side arrive/grant counters (no collective)",
           "ms_per_frame": tput, "mrays": W * H / tput / 1e3,
           "schedule": "two streams (two frames in flight per GPU)" if b["ms_per_frame_two_streams"] <= b["ms_per_frame"]
                       else "one stream (one frame in flight per GPU)",
           "ms_per_frame_latency": min(v["ms_per_frame"] for v in per_mode.values()),
           "ms_per_frame_1gpu": t1_pipe, "ms_per_frame_1gpu_latency": t1_lat,
           "speedup_vs_n1": t1_pipe / tput,
           "speedup_vs_n1_latency": t1_lat / min(v["ms_per_frame"] for v in per_mode.values()),
           "verified_bit_identical": verified,
           "limiting_kernel": {"name": b["kernel_names"][dom], "slowest_rank_ms": kmax[dom],
                               "per_rank_ms": [r[dom] for r in k],
                               "frame_minus_kernels_ms": b["ms_per_frame"] - sum(kmax)},
           "by_mode": {f"{m[0]}" + ("" if m[1] == "stores" else "_copy"):
                       {"ms_per_frame_latency": v["ms_per_frame"], "ms_per_frame_two_streams": v["ms_per_frame_two_streams"],
                        "kernels": v["kernel_names"], "kernels_ms_per_rank": v["kernels_ms_per_rank"]}
                       for m, v in per_mode.items()},
           "single_gpu_by_mode": {str(m): {"ms_per_frame_latency": v[0], "ms_per_frame_two_streams": v[1]}
                                  for m, v in single.items()},
           "e2e": {"ms_per_frame": e2e_ms, "mrays": W * H / e2e_ms / 1e3, "d2h_bytes_per_frame": W * H * 12,
                   "verified_bit_identical": host_verified,
                   "api": "rtgs.sharding.HostFrame: every rank DMAs its own stripes into one shared page-locked host "
                          "image over its own PCIe link, flags in the same shared memory; rank 0 collects every frame"}}
    return res


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from rtgs.synthetic import CONFIGS, make_scene
    arrays, n_g, seed, sh_deg, (W, H), n_views, orbit_phi, what = load_config(args.config, args.h_target)
    config = {"workload": f"{what}, {W}x{H}, fov 60, orbit r=2.2, depth {DEPTH}, t_cut {T_CUT}; "
                          f"{n_views}-view orbit, view (step*N+rank)%{n_views}",
              "gaussians": n_g, "sh_degree": sh_deg, "resolution": [W, H], "depth": DEPTH,
              "sharding": "camera views (scene replicated, no collective; at N > 1 every rank's kernels store their "
                          "frame into GPU 0's memory over NVLink and GPU 0 waits for the arrival counters)",
              "l2": "inputs larger than L2 (packed scene 528 MB > 126 MB) and a new view every step"}

    # ------------------------------------------------------------------ reference arm (CPU port)
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs writes the CUDA path's frames (--impl ours)")
        if rank != 0:
            return 0
        focal, views = make_views(W, H, n_views, orbit_phi)
        # bounded sample: every 4th column and row (1/16 of the rays) keeps 100 steps within ~1 minute of CPU time
        stride = args.cpu_stride or (4 if W * H <= 1920 * 1080 else 8)
        r = cpu_leg(args.config, arrays, W, H, focal, views, args.steps, args.warmup, stride)
        line = {"impl": "reference", "metric": "Mrays/s", "value": r["mrays"], "unit": "Mrays/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["mrays"], "unit": "Mrays/s", "cores": r["cores"], "kind": "port",
                                 "sample": r["sample"]},
                "e2e": {"value": r["mrays"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0,
                "note": "the reference is Python+Taichi and cannot run here; this is oracle/ref_cpu.cpp, a C++/OpenMP "
                        "port with the reference's algorithm shape, on the host cores"}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (CUDA)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the render path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from rtgs.camera import Camera
    from rtgs.ray_tracer import RayTracer
    from rtgs.scene import Scene

    if args.h_target is not None:
        config["workload"] += f" [diagnostic: h_target {args.h_target}]"
    if args.outliers > 0:
        rng = np.random.default_rng(99)
        arrays["pos"][:args.outliers] = (rng.uniform(-1, 1, (args.outliers, 3)) * 4000.0).astype(np.float32)
        config["workload"] += f" [diagnostic: {args.outliers} outliers at ~4000 scene radii]"
    if args.morton_bits == 63:
        config["workload"] += " [LBVH with 63-bit Morton codes]"
    focal, views = make_views(W, H, n_views, orbit_phi)
    t0 = time.perf_counter()
    scene = Scene(device=local_rank, morton_bits=args.morton_bits or "auto").from_arrays(
        arrays["pos"], arrays["rot"], arrays["scale"], arrays["color"], arrays["opacity"], arrays["sh"])
    torch.cuda.synchronize()
    build_ms = 1e3 * (time.perf_counter() - t0)
    cam = Camera(views[0][0], views[0][1], (W, H), (focal, focal), device=local_rank)
    rt = RayTracer((W, H), scene, cam, t_cut=T_CUT)
    out = torch.empty((W, H, 3), dtype=torch.float32, device="cuda")
    base_mode = scene.render_mode
    bvh_build_ms, morton_bits = scene.build_ms, scene.morton_bits
    kernel_names = [k or "-" for k in scene.kernel_names]
    launches_per_frame = sum(1 for k in scene.kernel_names if k)

    peer = None
    if world > 1:
        # SURVEY.md 8(d): the multi-GPU frame time ends with the framebuffers resident on GPU 0.  Slot r of the
        # peer-mapped buffer receives rank r's frame straight from its render kernels' stores.
        from rtgs.sharding import PeerFrame
        peer = PeerFrame(W, H, rank, world, local_rank, dist, slots=world, buffers=2)

    def set_view(step):
        v = (step * world + rank) % n_views
        cam.position, cam.rotation = views[v]
        return v

    def render_step():
        if peer is None:
            rt.render_device(DEPTH, out=out)
            return
        rt.render_device(DEPTH, out=peer.begin(scene, slot=rank))
        if rank == 0:
            peer.wait()          # all `world` frames of this step are in GPU 0's memory
            peer.release()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # stats pass (untimed): kbar, hit fraction, traversal counters for the timed views (whole frames)
    agg = {}
    stack_hw = [0, 0, 0]
    for s in range(min(args.steps, n_views)):
        set_view(s)
        rt.render_device(DEPTH, out=out, collect_stats=True)
        for k, v in rt.last_stats.items():
            agg[k] = agg.get(k, 0) + v
        stack_hw = [max(a, rt.last_stats[k]) for a, k in zip(stack_hw, ("max_lists_stack", "max_fused_stack", "max_group_list"))]
    tree_depth = scene.get_option("tree_depth")
    kbar = agg["layers"] / agg["rays"]
    bytes_ray = 16 + kbar * (64 + (192 if sh_deg > 0 else 0))

    for s in range(args.warmup):
        set_view(s)
        render_step()
    barrier()
    gathered_ok = None
    if peer is not None:
        # untimed check of the gather: slot r on GPU 0 == what GPU 0 renders itself for rank r's view
        set_view(0)
        render_step()
        barrier()
        if rank == 0:
            got = [peer.frame(r).clone() for r in range(world)]
            gathered_ok = True
            for r in range(world):
                cam.position, cam.rotation = views[r % n_views]
                gathered_ok = gathered_ok and bool(torch.equal(rt.render_device(DEPTH, out=out), got[r]))
            torch.cuda.synchronize()
        barrier()
    timed_frames = min(args.steps, 4096)
    scene.set_option("kernel_timing", timed_frames)   # events around every kernel of the timed steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    barrier()
    e_beg.record()
    for s in range(args.steps):
        set_view(s)
        ev[s][0].record()
        render_step()
        ev[s][1].record()
        launches += launches_per_frame
    e_end.record()
    barrier()
    # the last step's frame, read back untimed; the two-stream loop below renders the same steps, but both streams
    # store into the same buffer, so what it leaves there need not be one step's frame
    last_frames = None
    if args.dump_outputs:
        if rank == 0:
            last_frames = ({"frame": out.cpu().numpy()} if peer is None else
                           {f"frame_rank{r}": peer.frame(r).cpu().numpy() for r in range(world)})
        # the last step released its peer buffer, so the other ranks' next frames may already store into it:
        # hold them until rank 0 has read it back
        barrier()
    serial_ms = e_beg.elapsed_time(e_end)
    kern_ms = [a.elapsed_time(b) for a, b in ev]
    per_kernel = scene.read_kernel_times(timed_frames).astype(np.float64).mean(axis=0)   # ms of the frame's launches
    scene.set_option("kernel_timing", 0)

    # The throughput figure: the same K steps with frames alternating on two streams.  Frames on different streams
    # use separate frame scratch in the library (csrc/render.cu), so the head of step s+1 (its traversal kernel)
    # fills the SMs that the tail of step s leaves idle - the way the sweep API (render_async) runs.  Device-timed
    # with events on the default stream around both streams' work.
    ts = TwoStreams(torch)
    for s in range(args.warmup):
        set_view(s)
        with ts.stream(s):
            render_step()
    barrier()
    e0 = ts.begin()
    for s in range(args.steps):
        set_view(s)
        with ts.stream(s):
            render_step()
    e1 = ts.end()
    barrier()
    total_ms = e0.elapsed_time(e1)

    # end-to-end: public API call with host buffers (camera in, image out on the host), every rank its own frames
    def blocking(n):
        for s in range(n):
            set_view(s)
            rt.render(DEPTH)

    def pipelined(n, fmt="f32"):
        # the sweep API: every step still uploads its camera and delivers its image to pinned host memory, but
        # two frames are in flight (RayTracer.render_async), so step s+1 renders while step s is copied out.
        # Every image is collected inside the timed region.
        prev = None
        for s in range(n):
            set_view(s)
            cur = rt.render_async(DEPTH, fmt=fmt)
            if prev is not None:
                prev.result()
            prev = cur
        if prev is not None:
            prev.result()

    def wall(fn, n):
        fn(min(args.warmup, 3))
        barrier()
        t0 = time.perf_counter()
        fn(n)
        barrier()
        return time.perf_counter() - t0

    e2e_sync_s = wall(blocking, args.steps)
    e2e_pipe_s = wall(pipelined, args.steps)
    # opt-in compact delivery (the frame is still rendered in float32; 4 instead of 12 bytes per pixel cross PCIe)
    e2e_rgba8_s = wall(lambda n: pipelined(n, "rgba8"), args.steps)
    # the sampler has been running through all timed loops (device-timed steps and both end-to-end loops)
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "device-timed steps + end-to-end loops"
    # untimed repeat with the library's per-kernel events switched on: what the kernels cost in the pipelined mode
    scene.set_option("kernel_timing", timed_frames)
    pipelined(timed_frames)
    e2e_kernels = scene.read_kernel_times(timed_frames).astype(np.float64).mean(axis=0)
    scene.set_option("kernel_timing", 0)

    total_ms, serial_ms, e2e_pipe_s, e2e_sync_s, e2e_rgba8_s, kern_mean, *pk = allmax(
        dist, torch, [total_ms, serial_ms, e2e_pipe_s, e2e_sync_s, e2e_rgba8_s, float(np.mean(kern_ms)), *per_kernel.tolist()])
    per_kernel = np.asarray(pk)

    # ------------------------------------------------------------------ strong scaling: tile-sharded frames
    tiles = tiles4 = None
    tile_modes = [int(m) for m in args.tile_modes.split(",")]
    if not args.no_tiles:
        tiles = measure_tiles(torch, dist, rank, world, local_rank, scene, rt, cam, views, W, H,
                              min(args.steps, 128), args.warmup, barrier, tile_modes)
        scene.set_option("render_mode", base_mode)
    if (world >= 8 or args.config4) and not args.no_tiles and args.config == "1m_deg3_1080p":
        # BASELINE config 4: 3 M Gaussians, 3840x2160, tiles over all GPUs
        n4, seed4, deg4, (W4, H4) = CONFIGS["3m_deg3_2160p"]
        del rt, cam
        scene._release()
        a4 = make_scene(n4, seed4, deg4)
        focal4, views4 = make_views(W4, H4)
        scene4 = Scene(device=local_rank).from_arrays(a4["pos"], a4["rot"], a4["scale"], a4["color"], a4["opacity"], a4["sh"])
        cam4 = Camera(views4[0][0], views4[0][1], (W4, H4), (focal4, focal4), device=local_rank)
        rt4 = RayTracer((W4, H4), scene4, cam4, t_cut=T_CUT)
        tiles4 = measure_tiles(torch, dist, rank, world, local_rank, scene4, rt4, cam4, views4, W4, H4,
                               min(args.steps, 32), min(args.warmup, 3), barrier, tile_modes)
        if tiles4 is not None:
            tiles4["workload"] = f"synthetic {n4} random Gaussians, SH degree {deg4}, seed {seed4}, {W4}x{H4}"

    if rank == 0:
        rays_step = W * H * world
        value = rays_step * args.steps / (total_ms * 1e-3) / 1e6
        e2e_s = min(e2e_pipe_s, e2e_sync_s)
        e2e_val = rays_step * args.steps / e2e_s / 1e6
        peak, peak_src = load_peak()
        dom = int(np.argmax(per_kernel))
        dom_ms = float(per_kernel[dom])
        rays_launch = W * H                                 # rays one launch of the kernel processes
        achieved = rays_launch * bytes_ray / (dom_ms * 1e-3) / 1e9
        step_ms = float(per_kernel.sum())
        kernels = [{"kernel": kernel_names[k], "ms": float(per_kernel[k]), "share": float(per_kernel[k] / step_ms)}
                   for k in range(len(kernel_names)) if kernel_names[k] != "-"]
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak",
            "timing": "K steps alternating on two CUDA streams (two frames in flight per GPU), CUDA events on the "
                      "default stream around both, max over ranks; serial_* = the same K steps on one stream",
            "serial_value": rays_step * args.steps / (serial_ms * 1e-3) / 1e6, "serial_ms_per_step": serial_ms / args.steps,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_val, "unit": "Mrays/s", "h2d_bytes_per_step": 44 * world,
                    "d2h_bytes_per_step": W * H * 3 * 4 * world,
                    "ms_per_step": 1e3 * e2e_s / args.steps,
                    "api": ("RayTracer.render_async()/result(): two frames in flight, every image collected"
                            if e2e_pipe_s <= e2e_sync_s else "RayTracer.render() per step (blocking)") +
                           " [the faster of the two loops; both are reported]",
                    "pipelined_value": rays_step * args.steps / e2e_pipe_s / 1e6,
                    "sync_value": rays_step * args.steps / e2e_sync_s / 1e6,
                    "sync_api": "RayTracer.render() per step (blocking)",
                    "compact": {"format": "rgba8", "value": rays_step * args.steps / e2e_rgba8_s / 1e6,
                                "d2h_bytes_per_step": W * H * 4 * world,
                                "api": "RayTracer.render_async(fmt='rgba8'): same float32 render, the image is clipped "
                                       "and rounded to 8 bits per channel on the device before the DMA (opt-in; "
                                       "not the parity path, not the headline)"},
                    "kernels_ms": [round(float(v), 5) for v in e2e_kernels]},
            "gpu_launches": launches,
            "render_mode": base_mode,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": load_traffic(kernel_names[dom]), "peak_source": peak_src,
                         "kernel": kernel_names[dom], "kernel_ms": dom_ms, "step_ms": kern_mean,
                         "bytes_per_ray": bytes_ray, "kbar": kbar,
                         "note": "algorithmic bytes assume zero reuse between rays; neighbouring rays share "
                                 "Gaussians through L1/L2, so achieved may exceed what DRAM moved (see traffic)"},
            "kernels": kernels,
            "clocks": clocks,
            "scene_stats": {"hit_fraction": agg["rays_hit"] / agg["rays"], "kbar": kbar,
                            "child_boxes_tested_per_ray": agg["nodes_tested"] / agg["rays"],
                            "candidates_per_tile": agg["candidates"] / max(agg["tiles"], 1),
                            "pair_tests_per_ray": agg["pair_tests"] / agg["rays"],
                            "f64_refinements_per_Mray": 1e6 * agg["f64_refinements"] / agg["rays"],
                            "traversal_steps_per_tile": agg["traversal_steps"] / max(agg["tiles"], 1),
                            "insert_rounds_per_tile": agg["insert_rounds"] / max(agg["tiles"], 1),
                            "useful_candidates_per_tile": agg["useful_candidates"] / max(agg["tiles"], 1),
                            "fallback_tiles": agg["fallback_tiles"],
                            "stack_high_water": {"lists": stack_hw[0], "fused": stack_hw[1], "group_list": stack_hw[2],
                                                 "capacity": [256, 512, 960], "tree_depth": tree_depth}},
            "bvh_build_ms": bvh_build_ms,            # device time of the LBVH build kernels
            "morton_bits": morton_bits,
            "scene_load_ms": build_ms,               # wall: upload of the arrays + build (+ CUDA start-up on first use)
        }
        if peer is not None:
            line["gathered_on_gpu0"] = {"verified_bit_identical": gathered_ok,
                                        "how": "peer stores from every rank's render kernels + device-side arrival "
                                               "counters; the device-timed value includes rank 0's wait for them"}
        if tiles is not None:
            line["tiles"] = tiles
        if tiles4 is not None:
            line["tiles_config4"] = tiles4
        if world == 1 and not args.no_cpu_baseline:
            stride = args.cpu_stride or (4 if W * H <= 1920 * 1080 else 8)
            r = cpu_leg(args.config, arrays, W, H, focal, views, min(args.steps, 32), 1, stride)   # ~10-20 s of CPU work
            line["cpu_baseline"] = {"value": r["mrays"], "unit": "Mrays/s", "cores": r["cores"], "kind": "port",
                                    "steps": r["steps"], "sample": r["sample"]}
        else:
            line["cpu_baseline"] = None
        if last_frames is not None:
            dump_outputs(args.dump_outputs, last_frames)
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
