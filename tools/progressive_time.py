#!/usr/bin/env python3
"""Time-to-image of progressive rendering (Context.progressive) against one-shot nrrt_render on the benchmark workload:
configs 3 (Cornell box) and 4 (Utah teapot) at 1920x1080, 1024 spp, depth 50, AUTO mode.  Schedules, alternated within
each repetition: one-shot, progressive in 1 pass, in 4 passes (256 / 512 / 768 / 1024 samples) and one pass per chunk.
Each is timed on the host from the first launch to the f32 image in host memory (the one-shot render copies it back
itself; a progressive run ends with image()), and Mrays/s = closest-hit queries / that time.  Every progressive image
is checked to be the one-shot image bit for bit.  The device name and power limit go at the top of the log.

Usage: python tools/progressive_time.py [--reps 3] [--out FILE]"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nr_ray_tracer_b200 import _abi as A  # noqa: E402
from nr_ray_tracer_b200 import api  # noqa: E402
from nr_ray_tracer_b200.scene_config import CameraConfig, load_scene  # noqa: E402

CONFIGS = [("C3", "scenes/cornell-box-scene.json"), ("C4", "scenes/utah-teapot-scene.json")]
W, H, SPP, DEPTH = 1920, 1080, 1024, 50


def device_line() -> str:
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the name alone still says what the numbers were measured on
        q = f"power limit not read: {e}"
    return f"device: {name}; power limit, max SM clock: {q}"


def run_one_shot(ctx, cam):
    t0 = time.perf_counter()
    img, st = ctx.render(cam, seed=0, mode=A.MODE_AUTO)
    return time.perf_counter() - t0, img, st["segments"], 1


def run_progressive(ctx, cam, targets):
    t0 = time.perf_counter()
    segs = 0
    with ctx.progressive(cam, seed=0, mode=A.MODE_AUTO) as p:
        for t in targets:
            segs += p.render(t)["segments"]
        img = p.image()
    return time.perf_counter() - t0, img, segs, len(targets)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the log here")
    args = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    os.chdir(ROOT)
    ctx = api.Context(0)
    log(device_line())
    log(f"workload: {W}x{H}, {SPP} spp, depth {DEPTH}, MODE_AUTO, seed 0; {args.reps} repetitions, schedules alternated; "
        "time = host clock from the call to the f32 image in host memory")
    starts = api.chunk_starts(SPP, W * H)
    schedules = [("one-shot nrrt_render", None), ("progressive, 1 pass", [SPP]),
                 ("progressive, 4 passes", [256, 512, 768, 1024]),
                 (f"progressive, 1 pass per chunk ({len(starts) - 1})", starts[1:])]
    for cfg, path in CONFIGS:
        g = load_scene(path, camera_override=CameraConfig(width=W, height=H, samples_per_pixel=SPP, ray_max_bounces=DEPTH))
        hs = api.HostScene(g)
        ctx.upload(hs)
        cam = api.camera_build(g.camera.to_builder_config())
        _, ref, _, _ = run_one_shot(ctx, cam)  # warm-up (module load, scratch allocation)
        times = {label: [] for label, _ in schedules}
        segs = {}
        for _rep in range(args.reps):
            for label, targets in schedules:
                dt, img, s, n = run_one_shot(ctx, cam) if targets is None else run_progressive(ctx, cam, targets)
                assert np.array_equal(img, ref), (cfg, label)
                times[label].append(dt)
                segs[label] = s
        base = statistics.median(times[schedules[0][0]])
        log(f"\n{cfg} ({path}): {segs[schedules[0][0]]} segments per image; every progressive image == one-shot bit for bit")
        log(f"  {'schedule':42s} {'median s':>9s} {'min s':>8s} {'max s':>8s} {'Mrays/s':>9s} {'vs one-shot':>12s}")
        for label, _ in schedules:
            t = times[label]
            med = statistics.median(t)
            log(f"  {label:42s} {med:9.3f} {min(t):8.3f} {max(t):8.3f} {segs[label] / med / 1e6:9.1f} "
                f"{100.0 * (med / base - 1.0):+11.2f}%")
        del hs
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
