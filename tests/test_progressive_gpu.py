"""Progressive rendering on the GPU (nrrt_accum_*, Context.progressive, Scene.render_progressive, --preview-every): a
frame rendered in passes of whole chunks ends on nrrt_render's image bit for bit, whatever the passes, and every image
on the way is the oracle's render over the chunks done so far."""
import os
import subprocess

import numpy as np
import pytest

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200 import api
from oracle import oracle as O
from tests.scenes_util import load
from tests.test_gpu_parity import _moving_scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = [A.MODE_WAVEFRONT, A.MODE_MEGAKERNEL, A.MODE_FUSED, A.MODE_POOL, A.MODE_AUTO]
SCENES = ["cornell-box-scene.json", "utah-teapot-scene.json", "spheres.toml", "moving"]


def _graph(name, **cam):
    if name == "moving":
        g = _moving_scene(True)
        for k, v in cam.items():
            setattr(g.camera, k, v)
        return g
    return load(name, **cam)


def _setup(ctx, name, **cam):
    g = _graph(name, **cam)
    hs = api.HostScene(g)
    ctx.upload(hs)
    return g, hs, api.camera_build(g.camera.to_builder_config())


def _progressive(ctx, cam, targets, **kw):
    """Renders to each target in turn; returns (final image, [(samples done, image, stats)])."""
    passes = []
    with ctx.progressive(cam, **kw) as p:
        for t in targets:
            st = p.render(t)
            passes.append((p.samples, p.image(), st))
    return passes[-1][1], passes


@pytest.mark.parametrize("name", SCENES)
def test_final_image_is_the_one_shot_image(gpu_ctx, name):
    W, H, spp = 64, 36, 40
    g, hs, cam = _setup(gpu_ctx, name, width=W, height=H, samples_per_pixel=spp, ray_max_bounces=10)
    starts = api.chunk_starts(spp, W * H)
    assert starts == list(range(0, spp + 1, 2))  # 20 two-sample chunks at this size
    schedules = {"one pass": [spp], "per chunk": starts[1:], "[1 chunk, rest]": [starts[1], spp],
                 "off-boundary targets (round up)": [1, 5, 11, 39]}
    for mode in MODES:
        ref, st = gpu_ctx.render(cam, seed=9, mode=mode)
        for label, targets in schedules.items():
            img, passes = _progressive(gpu_ctx, cam, targets, seed=9, mode=mode)
            assert np.array_equal(img, ref), (name, mode, label)
            assert [s for s, _, _ in passes] == [min(s for s in starts if s >= t) for t in targets]
            assert sum(p[2]["paths"] for p in passes) == st["paths"] == W * H * spp
            assert sum(p[2]["segments"] for p in passes) == st["segments"], (name, mode, label)
            assert all(p[2]["mode"] == st["mode"] for p in passes if p[2]["paths"])
    del hs


@pytest.mark.parametrize("name", ["cornell-box-scene.json", "utah-teapot-scene.json"])
def test_every_intermediate_image_is_the_oracle_s_render_of_the_chunks_done(gpu_ctx, name):
    W, H, spp = 48, 27, 30
    g, hs, cam = _setup(gpu_ctx, name, width=W, height=H, samples_per_pixel=spp, ray_max_bounces=50)
    starts = api.chunk_starts(spp, W * H)
    assert len(starts) - 1 == 15
    osc, ocam = O.OracleScene(g), O.camera_build(g.camera.to_builder_config())
    prev_segments = 0
    with gpu_ctx.progressive(cam, seed=4) as p:
        assert p.samples == 0
        with pytest.raises(api.NrrtError):  # nothing to show before the first pass
            p.image()
        for k in range(1, len(starts)):
            st = p.render(starts[k])
            assert p.samples == starts[k]
            ref, cnt = osc.render_chunked(ocam, starts[:k + 1], seed=4)
            assert np.array_equal(p.image(), ref), (name, k)
            assert st["segments"] == cnt["segments"] - prev_segments, (name, k)
            assert st["paths"] == W * H * (starts[k] - starts[k - 1]) and cnt["paths"] == W * H * starts[k]
            prev_segments = cnt["segments"]
    del hs


def test_partitions_assemble_to_the_one_shot_image(gpu_ctx):
    import torch
    W, H, spp = 64, 37, 6
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=spp)
    full, _ = gpu_ctx.render(cam, seed=5)
    targets = [2, 3, spp]
    for world in (2, 3, 8):
        for R in (1, 8):
            asm = np.full_like(full, np.nan)
            for rank in range(world):
                rows = np.array([y for y in range(H) if (y // R) % world == rank], dtype=np.int64)
                assert len(rows) == api.owned_rows(H, rank, world, R)
                with gpu_ctx.progressive(cam, seed=5, rank=rank, world=world, rows_per_block=R) as p:
                    for t in targets:
                        st = p.render(t)
                        assert st["pixels"] == len(rows) * W
                    assert p.samples == spp
                    p.image(out=asm)
                    packed = p.image(packed=True)
                    assert packed.shape == (len(rows), W, 3)
                    assert np.array_equal(packed, full[rows]), (world, R, rank)
                    if len(rows):
                        dev = torch.full((len(rows), W, 3), float("nan"), device="cuda")
                        p.image(packed=True, out_device_ptr=dev.data_ptr())
                        assert np.array_equal(dev.cpu().numpy(), full[rows])
                        devf = torch.full((H, W, 3), float("nan"), device="cuda")
                        p.image(out_device_ptr=devf.data_ptr())
                        assert np.array_equal(devf.cpu().numpy()[rows], full[rows])
                    n, sums = p.state()
                    assert n == spp and sums.shape == (len(rows), W, 3)
                if world == 8 and R == 8 and rank >= 5:
                    assert len(rows) == 0  # 5 row-blocks: ranks 5..7 own nothing and still run every pass
            assert np.array_equal(asm, full), (world, R)
    del hs


def test_resume_on_a_fresh_context_and_validation(gpu_ctx):
    W, H, spp = 64, 36, 40
    g, hs, cam = _setup(gpu_ctx, "utah-teapot-scene.json", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=8)
    starts = api.chunk_starts(spp, W * H)
    assert starts[5] + 1 not in starts
    ref, _ = gpu_ctx.render(cam, seed=3)
    with gpu_ctx.progressive(cam, seed=3) as p:
        p.render(starts[2])
        p.render(starts[5])
        done, sums = p.state()
        mid = p.image()
    assert done == starts[5]
    ctx2 = api.Context(0)
    try:
        hs2 = api.HostScene(g)
        ctx2.upload(hs2)
        with ctx2.progressive(cam, seed=3) as q:
            for bad in (starts[5] + 1, spp + 1, 10 ** 6):
                with pytest.raises(api.NrrtError) as e:
                    q.restore(bad, sums)
                assert e.value.code == A.ERR_INVALID
            q.restore(done, sums)
            assert q.samples == done
            assert np.array_equal(q.image(), mid)
            q.render(spp)
            assert np.array_equal(q.image(), ref)
            # replacing the scene invalidates the frame
            ctx2.upload(hs2)
            for call in (lambda: q.render(spp), q.image, q.state, lambda: q.restore(done, sums)):
                with pytest.raises(api.NrrtError) as e:
                    call()
                assert e.value.code == A.ERR_NO_SCENE
        del hs2
    finally:
        ctx2.close()
    del hs


def test_depth_zero_is_black_in_every_pass(gpu_ctx):
    W, H, spp = 32, 18, 8
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=0)
    ref, _ = gpu_ctx.render(cam)
    img, passes = _progressive(gpu_ctx, cam, api.chunk_starts(spp, W * H)[1:])
    assert all(not im.any() for _, im, _ in passes)
    assert np.array_equal(img, ref)
    del hs


def test_scene_render_progressive_yields_passes_ending_on_render(gpu_ctx):
    from nr_ray_tracer_b200.scene_config import CameraConfig
    s = api.Scene.load("scenes/cornell-box-scene.json",
                       camera_override=CameraConfig(width=48, height=27, samples_per_pixel=9), ctx=gpu_ctx)
    ref = s.render(seed=2)
    starts = api.chunk_starts(9, 48 * 27)
    got = list(s.render_progressive(seed=2))
    assert [n for n, _ in got] == starts[1:]
    assert np.array_equal(got[-1][1], ref)
    got4 = list(s.render_progressive(every=4, seed=2))
    assert [n for n, _ in got4] == [min(x for x in starts if x >= t) for t in (4, 8, 9)]
    assert np.array_equal(got4[-1][1], ref)


@pytest.mark.parametrize("name", ["cornell-box-scene.json", "utah-teapot-scene.json"])
def test_benchmark_workload_in_four_passes_is_the_one_shot_image(gpu_ctx, name):
    W, H, spp = 1920, 1080, 1024
    g, hs, cam = _setup(gpu_ctx, name, width=W, height=H, samples_per_pixel=spp, ray_max_bounces=50)
    ref, st = gpu_ctx.render(cam, seed=0, mode=A.MODE_AUTO)
    img, passes = _progressive(gpu_ctx, cam, [256, 512, 768, 1024], seed=0, mode=A.MODE_AUTO)
    assert np.array_equal(img, ref), name
    assert sum(p[2]["segments"] for p in passes) == st["segments"]
    del hs


def test_cli_preview_every_writes_the_same_final_file(gpu_ctx, tmp_path):
    from nr_ray_tracer_b200 import build as B
    B.build()
    base = [B.CLI, "render", "scenes/cornell-box-scene.json", "-W", "96", "-H", "54", "--samples-per-pixel", "20",
            "--seed", "5"]
    plain, prog = tmp_path / "plain.png", tmp_path / "prog.png"
    r = subprocess.run(base + ["-o", str(plain)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    r = subprocess.run(base + ["-o", str(prog), "--preview-every", "6", "-v"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert prog.read_bytes() == plain.read_bytes()
    starts = api.chunk_starts(20, 96 * 54)
    done = [int(line.split()[1]) for line in r.stderr.splitlines() if line.startswith("pass: ")]
    assert done == [min(s for s in starts if s >= min(t, 20)) for t in (6, 12, 18, 24)]
    assert all(d in starts for d in done)
    assert not [f for f in os.listdir(tmp_path) if ".tmp" in f]  # previews went through a renamed temporary file
    # the create-new check still holds
    r = subprocess.run(base + ["-o", str(prog), "--preview-every", "6"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode != 0 and prog.read_bytes() == plain.read_bytes()
