#!/usr/bin/env python3
"""Denoising cost and quality on one GPU.

Cost: the guide pass (nrrt_accum_aov, 16 samples per pixel) and the filter (nrrt_accum_denoise, 5 iterations) at
1920x1080 and 3840x2160 on C2a earth, C3 Cornell box and C4 Utah teapot, next to the one-shot render of the config at
1920x1080 (C2a 256 spp, C3 / C4 1024 spp, depth 50 for C3 / C4).  Outputs go to device buffers, so no PCIe copy is timed.
Each call is timed on the host around the library call, which ends in a device synchronise: the guide pass on a fresh
frame each repetition (its guides are computed on first use), the filter repeatedly on one frame.  Medians.

Quality: RMSE against a 4096-spp render (seed 1) of the same scene and size, 400x225, depth 10, of the noisy image and
the denoised one (defaults: 5 iterations, sigma_color 4, 16 guide samples) after 16, 64 and 256 spp (seed 2, one pass).
tests/test_denoise_gpu.py asserts the 64-spp ratio of these same renders.

The device name and power limit go at the top of the log.

Usage: python tools/denoise_time.py [--reps 5] [--out FILE] [--skip-cost] [--skip-quality]"""
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

COST = [("C2a", "scenes/earth.toml", 256, None), ("C3", "scenes/cornell-box-scene.json", 1024, 50),
        ("C4", "scenes/utah-teapot-scene.json", 1024, 50)]
SIZES = [(1920, 1080), (3840, 2160)]
QUALITY = [("Cornell", "scenes/cornell-box-scene.json"), ("earth", "scenes/earth.toml"),
           ("teapot", "scenes/utah-teapot-scene.json")]
QUALITY_SIZE, QUALITY_REF_SPP, QUALITY_SPP = (400, 225), 4096, [16, 64, 256]


def scene(ctx, path, W, H, spp, depth):
    g = load_scene(os.path.join(ROOT, path), base_dir=ROOT,
                   camera_override=CameraConfig(width=W, height=H, samples_per_pixel=spp, ray_max_bounces=depth))
    sc = api.Scene(g, ctx=ctx)
    return sc


def cost(ctx, log, reps):
    import torch
    log(f"cost: medians of {reps} (ms); guides = nrrt_accum_aov with 16 samples per pixel, filter = nrrt_accum_denoise "
        "with 5 iterations; one-shot = nrrt_render of the config at 1920x1080")
    log(f"{'config':6} {'size':>9} {'guides':>8} {'filter':>8} {'sum':>8} {'one-shot':>9} {'share':>7}")
    for name, path, spp, depth in COST:
        one_shot = None
        for W, H in SIZES:
            sc = scene(ctx, path, W, H, spp, depth)
            cam = sc.camera
            if (W, H) == SIZES[0]:
                ctx.render(cam, seed=0)  # warm-up
                ts = []
                for _ in range(2):
                    t0 = time.perf_counter()
                    ctx.render(cam, seed=0)
                    ts.append(time.perf_counter() - t0)
                one_shot = statistics.median(ts) * 1e3
            da = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
            dn = torch.empty_like(da)
            tg = []
            for r in range(reps + 1):
                with ctx.progressive(cam, seed=0) as p:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    p.aov(16, out_device_ptr=(da.data_ptr(), dn.data_ptr()))
                    if r:
                        tg.append(time.perf_counter() - t0)
            cam16 = A.Camera.from_buffer_copy(cam)
            cam16.samples_per_pixel = 16
            tf = []
            with ctx.progressive(cam16, seed=0, adaptive={"rel_error": 0.0}) as p:
                p.render(16)
                p.aov(16, out_device_ptr=(da.data_ptr(), dn.data_ptr()))
                for r in range(reps + 1):
                    t0 = time.perf_counter()
                    p.denoised(out_device_ptr=da.data_ptr())
                    if r:
                        tf.append(time.perf_counter() - t0)
            g_ms, f_ms = statistics.median(tg) * 1e3, statistics.median(tf) * 1e3
            log(f"{name:6} {W:>4}x{H:<4} {g_ms:8.2f} {f_ms:8.2f} {g_ms + f_ms:8.2f} {one_shot:9.1f} "
                f"{100 * (g_ms + f_ms) / one_shot:6.2f}%")
            del da, dn
            sc.host.close()


def rmse(x, ref):
    return float(np.sqrt(np.mean((x.astype(np.float64) - ref) ** 2)))


def quality_rows(ctx, path, spps=QUALITY_SPP):
    """(spp, noisy RMSE, denoised RMSE) against the 4096-spp render, as tests/test_denoise_gpu.py computes them."""
    W, H = QUALITY_SIZE
    sc = scene(ctx, path, W, H, QUALITY_REF_SPP, 10)
    ref, _ = ctx.render(sc.camera, seed=1)
    rows = []
    for spp in spps:
        cam = A.Camera.from_buffer_copy(sc.camera)
        cam.samples_per_pixel = spp
        with ctx.progressive(cam, seed=2, adaptive={"rel_error": 0.0}) as p:
            p.render(spp)
            rows.append((spp, rmse(p.image(), ref), rmse(p.denoised(), ref)))
    sc.host.close()
    return rows


def quality(ctx, log):
    W, H = QUALITY_SIZE
    log(f"quality: RMSE against {QUALITY_REF_SPP} spp (seed 1), {W}x{H}, depth 10; noisy and denoised (seed 2)")
    log(f"{'scene':8} {'spp':>5} {'noisy':>9} {'denoised':>9} {'ratio':>6}")
    for name, path in QUALITY:
        for spp, noisy, den in quality_rows(ctx, path):
            log(f"{name:8} {spp:5d} {noisy:9.5f} {den:9.5f} {den / noisy:6.3f}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the log here")
    ap.add_argument("--skip-cost", action="store_true")
    ap.add_argument("--skip-quality", action="store_true")
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(device_line())
    ctx = api.Context(0)
    if not args.skip_cost:
        cost(ctx, log, args.reps)
    if not args.skip_quality:
        quality(ctx, log)
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
