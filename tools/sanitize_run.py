#!/usr/bin/env python3
"""Small renders for compute-sanitizer (developer tool, GPU box): every kernel design on a 64x36 Cornell box, the
pooled and fused kernels on the teapot mesh and the sphere field, an adaptive frame in every design, the denoising
guides and filter (odd sizes: taps past every border), scenes whose
traversal stacks are full by construction (four instance levels, 65536 instances), a fixed-ray batch each.
  compute-sanitizer --tool memcheck  python tools/sanitize_run.py
  compute-sanitizer --tool racecheck python tools/sanitize_run.py"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nr_ray_tracer_b200 import _abi as A, api  # noqa: E402
from nr_ray_tracer_b200.scene_config import CameraConfig, load_scene  # noqa: E402
from tests import kat  # noqa: E402
from tools import instance_scenes as S  # noqa: E402

ctx = api.Context(0)
for name, modes in (("cornell-box-scene.json", (A.MODE_FUSED, A.MODE_POOL, A.MODE_WAVEFRONT, A.MODE_MEGAKERNEL)),
                    ("utah-teapot-scene.json", (A.MODE_FUSED, A.MODE_POOL)), ("spheres.toml", (A.MODE_FUSED, A.MODE_POOL)),
                    ("noise.toml", (A.MODE_POOL,))):
    g = load_scene("scenes/" + name, camera_override=CameraConfig(width=64, height=36, samples_per_pixel=2, ray_max_bounces=50))
    hs = api.HostScene(g)
    ctx.upload(hs)
    cam = api.camera_build(g.camera.to_builder_config())
    ref = None
    for m in modes:
        img, st = ctx.render(cam, seed=1, mode=m)
        ref = img if ref is None else ref
        assert np.array_equal(img, ref)
        print(name, A.MODE_NAMES[m], st["segments"], flush=True)
    rays = np.concatenate([kat.random_rays(g, 2000), kat.special_rays(g)[:500]])
    hits, _ = ctx.trace_rays(rays)
    print(name, "trace", int((hits["object"] != 0xFFFFFFFF).sum()), flush=True)
# adaptive frames in every design: the active-list decode, k_resolve_adaptive, the ordered compaction, the per-pixel
# maps, and a restore
g = load_scene("scenes/spheres.toml", camera_override=CameraConfig(width=64, height=36, samples_per_pixel=24, ray_max_bounces=50))
hs = api.HostScene(g)
ctx.upload(hs)
cam = api.camera_build(g.camera.to_builder_config())
ref = None
for m in (A.MODE_FUSED, A.MODE_POOL, A.MODE_WAVEFRONT, A.MODE_MEGAKERNEL):
    with ctx.progressive(cam, seed=1, mode=m, adaptive={"rel_error": 0.05, "min_samples": 2}) as p:
        passes = []
        while p.active:
            p.render(p.samples + 1)
            passes.append(p.active)
            if len(passes) == 3:
                p.restore(*p.state())
        img, err, n = p.image(), p.error_image(), p.sample_map()
    ref = (img, n) if ref is None else ref
    assert np.array_equal(img, ref[0]) and np.array_equal(n, ref[1])
    print("adaptive", A.MODE_NAMES[m], "active per pass", passes, "mean samples", float(n.mean()), flush=True)
# denoising: the guide pass (k_aov, on a partition too) and every filter iteration (k_denoise_*: the checked build
# bounds-checks each tap) on odd sizes, so that taps fall past every border at every spacing
for W, H in ((1, 1), (7, 3), (33, 17)):
    gd = load_scene("scenes/earth.toml", camera_override=CameraConfig(width=W, height=H, samples_per_pixel=6, ray_max_bounces=8))
    hs = api.HostScene(gd)
    ctx.upload(hs)
    cam_d = api.camera_build(gd.camera.to_builder_config())
    with ctx.progressive(cam_d, seed=1, adaptive={"rel_error": 0.0}) as p:
        p.render(p.samples_per_pixel)
        out = p.denoised(iterations=8, aov_samples=3)
    with ctx.progressive(cam_d, seed=1, world=3, rank=1, rows_per_block=1) as p:
        p.aov(2)
    print("denoise", W, H, "finite", bool(np.isfinite(out).all()), flush=True)
# stacks full by construction (tools/instance_scenes.py): four instance levels at max_stack 32, the LITE pool variant at
# its per-scene cap (binary stack 24), and 65536 instances (ids past 16 bits in the pooled kernel's chain words)
for name, g, runs in (("full_stack(32)", S.full_stack(32), ((A.MODE_FUSED, None), (A.MODE_POOL, "0"), (A.MODE_WAVEFRONT, None))),
                      ("lite_full_stack", S.lite_full_stack(), ((A.MODE_POOL, "1"), (A.MODE_FUSED, None))),
                      ("nested(4, spec)", S.nested(4, mesh="spec")[0], ((A.MODE_FUSED, None), (A.MODE_POOL, "0"))),
                      ("many_instances(65535)", S.many_instances(65535, 1, width=32, height=18, spp=1),
                       ((A.MODE_POOL, None), (A.MODE_FUSED, None)))):
    hs = api.HostScene(g)
    ctx.upload(hs)
    cam = api.camera_build(g.camera.to_builder_config())
    ref = None
    for m, lite in runs:
        os.environ.pop("NRRT_POOL_LITE", None)
        if lite is not None:
            os.environ["NRRT_POOL_LITE"] = lite
        img, st = ctx.render(cam, seed=1, mode=m)
        ref = img if ref is None else ref
        assert np.array_equal(img, ref)
        print(name, A.MODE_NAMES[m], "lite=" + str(lite), "max_stack", hs.desc.max_stack, st["segments"], flush=True)
    os.environ.pop("NRRT_POOL_LITE", None)
    hits, _ = ctx.trace_rays(np.concatenate([kat.random_rays(g, 2000), kat.aimed_rays(g, 2000)]))
    print(name, "trace", int((hits["object"] != 0xFFFFFFFF).sum()), flush=True)
print("sanitize_run done")
