#!/usr/bin/env python3
"""Adaptive sampling against one-shot nrrt_render and against plain progressive rendering with the same passes, on one
GPU at the configs' own sizes: C1 spheres (400x225, 100 spp), C2a earth (1920x1080, 256 spp), C3 Cornell box and C4
Utah teapot (1920x1080, 1024 spp, depth 50), AUTO mode, seed 0.

For tolerances rel_error in {0, 0.01, 0.03} (abs_error 0, the default min_samples: the first chunk boundary at or above
spp / 8) the adaptive frame runs Scene.render_adaptive's default schedule: passes ending at doubling chunk counts from
min_samples.  Plain progressive runs the same pass ends.  Each run is timed on the host from the first launch to the
f32 image in host memory; segments are the closest-hit queries the run made.  Checks: tolerance 0 gives the one-shot
image bit for bit, and at every tolerance a pixel that took every sample equals the one-shot pixel.  Also printed: the
fraction of pixels retired after each pass.  The device name and power limit go at the top of the log.

Usage: python tools/adaptive_time.py [--reps 2] [--out FILE]"""
import argparse
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nr_ray_tracer_b200 import _abi as A  # noqa: E402
from nr_ray_tracer_b200 import api  # noqa: E402
from nr_ray_tracer_b200.scene_config import CameraConfig, load_scene  # noqa: E402
from tools.progressive_time import device_line  # noqa: E402

CONFIGS = [("C1", "scenes/spheres.toml", 400, 225, 100, 50), ("C2a", "scenes/earth.toml", 1920, 1080, 256, None),
           ("C3", "scenes/cornell-box-scene.json", 1920, 1080, 1024, 50),
           ("C4", "scenes/utah-teapot-scene.json", 1920, 1080, 1024, 50)]
TOLERANCES = [0.0, 0.01, 0.03]


def pass_ends(spp, pixels):
    starts = api.chunk_starts(spp, pixels)
    k, out = starts.index(api.default_min_samples(spp, pixels)), []
    while k < len(starts) - 1:
        out.append(starts[k])
        k *= 2
    return out + [spp]


def run_one_shot(ctx, cam):
    t0 = time.perf_counter()
    img, st = ctx.render(cam, seed=0, mode=A.MODE_AUTO)
    return time.perf_counter() - t0, img, st["segments"], None


def run_passes(ctx, cam, targets, rel):
    """Plain progressive (rel None) or adaptive; returns (s, image, segments, retired fraction after each pass)."""
    t0 = time.perf_counter()
    segs, retired = 0, []
    ad = None if rel is None else {"rel_error": rel}
    with ctx.progressive(cam, seed=0, mode=A.MODE_AUTO, adaptive=ad) as p:
        total = cam.width * cam.height
        for t in targets:
            if ad is not None and not p.active:
                break
            segs += p.render(t)["segments"]
            if ad is not None:
                retired.append(1.0 - p.active / total if p.samples < cam.samples_per_pixel else None)
        img = p.image()
        dt = time.perf_counter() - t0
        if ad is not None:
            retired = (retired, p.sample_map())
    return dt, img, segs, retired


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the log here")
    args = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    os.chdir(ROOT)
    ctx = api.Context(0)
    log(device_line())
    log(f"MODE_AUTO, seed 0, abs_error 0, default min_samples; {args.reps} repetitions, runs alternated; time = host "
        "clock from the call to the f32 image in host memory")
    for cfg, path, W, H, spp, depth in CONFIGS:
        cc = dict(width=W, height=H, samples_per_pixel=spp)
        if depth is not None:
            cc["ray_max_bounces"] = depth
        g = load_scene(path, camera_override=CameraConfig(**cc))
        hs = api.HostScene(g)
        ctx.upload(hs)
        cam = api.camera_build(g.camera.to_builder_config())
        targets = pass_ends(spp, W * H)
        runs = [("one-shot nrrt_render", "one", None), (f"progressive, same {len(targets)} passes", "prog", None)] + \
               [(f"adaptive rel_error {t:g}", "ad", t) for t in TOLERANCES]
        _, ref, _, _ = run_one_shot(ctx, cam)  # warm-up (module load, scratch allocation) ...
        for _label, kind, rel in runs[1:]:      # ... of every run: the adaptive passes launch kernels of their own
            run_passes(ctx, cam, targets, rel if kind == "ad" else None)
        times = {label: [] for label, _, _ in runs}
        segs, extra = {}, {}
        for _rep in range(args.reps):
            for label, kind, rel in runs:
                if kind == "one":
                    dt, img, s, x = run_one_shot(ctx, cam)
                else:
                    dt, img, s, x = run_passes(ctx, cam, targets, rel if kind == "ad" else None)
                if kind == "ad":
                    full = x[1] == spp
                    assert np.array_equal(img[full], ref[full]), (cfg, label)
                    assert rel > 0 or full.all()
                else:
                    assert np.array_equal(img, ref), (cfg, label)
                times[label].append(dt)
                segs[label], extra[label] = s, x
        base = statistics.median(times[runs[0][0]])
        base_segs = segs[runs[0][0]]
        prog = statistics.median(times[runs[1][0]])
        log(f"\n{cfg} ({path}, {W}x{H}, {spp} spp, depth {cam.ray_max_bounces}): pass ends {targets}")
        log(f"  {'run':32s} {'median s':>9s} {'min s':>8s} {'max s':>8s} {'segments':>13s} {'segs':>7s} "
            f"{'vs one-shot':>12s} {'vs progressive':>15s}")
        for label, kind, _ in runs:
            t = times[label]
            med = statistics.median(t)
            log(f"  {label:32s} {med:9.3f} {min(t):8.3f} {max(t):8.3f} {segs[label]:13d} "
                f"{100.0 * segs[label] / base_segs:6.1f}% {100.0 * (med / base - 1.0):+11.2f}% "
                f"{100.0 * (med / prog - 1.0):+14.2f}%")
        for label, kind, rel in runs:
            if kind == "ad":
                fr, smap = extra[label]
                cells = ", ".join(f"{targets[i]}: {'done' if f is None else f'{100.0 * f:.1f}%'}" for i, f in enumerate(fr))
                log(f"  retired after each pass, {label}: {cells}; mean samples per pixel {smap.mean():.1f}")
        del hs
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
