"""Denoising on the GPU (nrrt_accum_aov, nrrt_accum_denoise, Progressive.aov / denoised, Scene.render_denoised,
--denoise): the guides are the oracle's bit for bit on every scene kind and partition, the filter is its float32 numpy
statement bit for bit on the handle's own state and guides, the result does not depend on the kernel design, and
nothing the frame already returned changes."""
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200 import api
from tests import aov_ref as AR
from tests import denoise_ref as D
from tests.scenes_util import load
from tests.test_gpu_parity import _moving_scene
from tools import instance_scenes as IS

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = [A.MODE_WAVEFRONT, A.MODE_MEGAKERNEL, A.MODE_FUSED, A.MODE_POOL, A.MODE_AUTO]
GUIDE_SCENES = ["cornell-box-scene.json", "utah-teapot-scene.json", "spheres.toml", "earth.toml", "noise.toml", "moving",
                "nested4"]


def _graph(name, **cam):
    if name == "moving":
        g = _moving_scene(True)
    elif name == "nested4":
        g, _ = IS.nested(4, mesh="inner", textured=True)
    else:
        return load(name, **cam)
    for k, v in cam.items():
        setattr(g.camera, k, v)
    return g


def _setup(ctx, name, **cam):
    g = _graph(name, **cam)
    hs = api.HostScene(g)
    ctx.upload(hs)
    return g, hs, api.camera_build(g.camera.to_builder_config())


def _filter_ref(p, iterations=5, sigma_color=4.0, aov_samples=None):
    """denoise_ref on the handle's own state and guides."""
    S, Q, N = p.state()
    starts = api.chunk_starts(p.samples_per_pixel, p.camera.width * p.camera.height)
    K = np.searchsorted(np.asarray(starts), N)
    assert (np.asarray(starts)[K] == N).all()
    C_, e2 = D.inputs(S, Q, N, K)
    albedo, normal = p.aov(aov_samples)
    return D.denoise(C_, e2, albedo, normal, iterations=iterations, sigma_color=sigma_color)


@pytest.mark.parametrize("name", GUIDE_SCENES)
def test_guides_are_the_oracle_s(gpu_ctx, name):
    W, H, spp = 64, 36, 24
    g, hs, cam = _setup(gpu_ctx, name, width=W, height=H, samples_per_pixel=spp, ray_max_bounces=6)
    with gpu_ctx.progressive(cam, seed=7) as p:
        for n in (None, 1, 5, spp):
            albedo, normal = p.aov(n)
            ra, rn = AR.oracle_aov(g, cam, 16 if n is None else n, seed=7)
            assert np.array_equal(albedo, ra), (name, n, np.argwhere(albedo != ra)[:4])
            assert np.array_equal(normal, rn), (name, n, np.argwhere(normal != rn)[:4])
        assert (np.abs(normal) > 0).any() and (albedo > 0).any()
    del hs


@pytest.mark.parametrize("world,rpb", [(2, 8), (3, 1), (8, 8)])
def test_guides_on_every_partition_and_layout(gpu_ctx, world, rpb):
    import torch
    W, H, spp = 37, 23, 6
    g, hs, cam = _setup(gpu_ctx, "earth.toml", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=4)
    ra, rn = AR.oracle_aov(g, cam, 4, seed=2)
    for rank in range(world):
        rows = api.owned_rows(H, rank, world, rpb)
        ys = [y for y in range(H) if (y // rpb) % world == rank]
        assert len(ys) == rows
        with gpu_ctx.progressive(cam, seed=2, rank=rank, world=world, rows_per_block=rpb) as p:
            fa, fn = p.aov(4)
            pa, pn = p.aov(4, packed=True)
            assert np.array_equal(fa[ys], ra[ys]) and np.array_equal(fn[ys], rn[ys]), rank
            other = [y for y in range(H) if y not in ys]
            assert (fa[other] == 0).all() and (fn[other] == 0).all()  # rows of other ranks untouched
            assert np.array_equal(pa, ra[ys]) and np.array_equal(pn, rn[ys]), rank
            for packed in (False, True):
                da = torch.zeros(((rows if packed else H), W, 3), dtype=torch.float32, device="cuda")
                dn = torch.zeros_like(da)
                p.aov(4, packed=packed, out_device_ptr=(da.data_ptr(), dn.data_ptr()))
                torch.cuda.synchronize()
                want_a, want_n = (pa, pn) if packed else (fa, fn)
                assert np.array_equal(da.cpu().numpy(), want_a) and np.array_equal(dn.cpu().numpy(), want_n)
    del hs


@pytest.mark.parametrize("W,H", [(1, 1), (7, 3), (33, 17), (400, 225)])
def test_filter_is_the_numpy_statement(gpu_ctx, W, H):
    spp = 48
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=8)
    with gpu_ctx.progressive(cam, seed=3, adaptive={"rel_error": 0.0, "min_samples": 0}) as p:
        p.render(spp)
        its = range(1, 9) if (W, H) == (33, 17) else [5]
        for it in its:
            out = p.denoised(iterations=it)
            ref = _filter_ref(p, iterations=it)
            assert np.array_equal(out, ref), (W, H, it, np.argwhere(out != ref)[:4])
        out = p.denoised(iterations=3, sigma_color=0.5, aov_samples=2)
        assert np.array_equal(out, _filter_ref(p, iterations=3, sigma_color=0.5, aov_samples=2))
    del hs


def test_filter_on_one_chunk_and_on_retired_pixels(gpu_ctx):
    # one chunk: K = 1 everywhere, no error estimate (v = +inf, colour weight 1)
    W, H = 64, 36
    g, hs, cam = _setup(gpu_ctx, "earth.toml", width=W, height=H, samples_per_pixel=1, ray_max_bounces=8)
    with gpu_ctx.progressive(cam, seed=1, adaptive={"rel_error": 0.0, "min_samples": 0}) as p:
        p.render(1)
        assert len(api.chunk_starts(1, W * H)) == 2
        out = p.denoised()
        assert np.isfinite(out).all() and np.array_equal(out, _filter_ref(p))
    # an adaptive frame whose pixels stopped at different sample counts
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=256, ray_max_bounces=8)
    with gpu_ctx.progressive(cam, seed=4, adaptive={"rel_error": 0.08, "abs_error": 0.002}) as p:
        starts = api.chunk_starts(256, W * H)
        for t in starts[3::3] + [256]:
            if p.active:
                p.render(t)
            out = p.denoised()
            assert np.array_equal(out, _filter_ref(p)), t
        N = p.state()[2]
        assert len(np.unique(N)) > 2, np.unique(N)
    del hs


def test_denoised_image_is_the_same_for_every_mode(gpu_ctx):
    import torch
    W, H, spp = 96, 54, 40
    g, hs, cam = _setup(gpu_ctx, "utah-teapot-scene.json", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=8)
    first = None
    for mode in MODES:
        with gpu_ctx.progressive(cam, seed=6, mode=mode, adaptive={"rel_error": 0.05}) as p:
            while p.active:
                p.render(p.samples + 1)
            out = p.denoised()
            d = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda")
            p.denoised(out_device_ptr=d.data_ptr())
            torch.cuda.synchronize()
            assert np.array_equal(d.cpu().numpy(), out)
        if first is None:
            first = out
        assert np.array_equal(out, first), mode
    del hs


def test_render_denoised_leaves_the_image_alone(gpu_ctx):
    W, H, spp = 80, 45, 32
    g = load("spheres.toml", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=8)
    sc = api.Scene(g, ctx=gpu_ctx)
    plain = sc.render(seed=11)
    image, den = sc.render_denoised(seed=11)
    assert np.array_equal(image, plain)
    assert den.shape == image.shape and np.isfinite(den).all() and not np.array_equal(den, image)
    with gpu_ctx.progressive(sc.camera, seed=11, adaptive={"rel_error": 0.0}) as p:
        p.render(spp)
        before = p.state()
        assert np.array_equal(p.denoised(), den)
        assert np.array_equal(p.image(), plain)  # denoising changed nothing the frame holds
        assert all(np.array_equal(a, b) for a, b in zip(p.state(), before))
    image2, den2 = sc.render_denoised(rel_error=0.05, seed=11, iterations=3)
    assert np.isfinite(den2).all()


def test_refusals(gpu_ctx):
    W, H, spp = 32, 18, 8
    g, hs, cam = _setup(gpu_ctx, "quads.toml", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=4)
    L = api.lib()
    out = np.zeros((H, W, 3), np.float32)
    ptr = out.ctypes.data

    def rc(p, **kw):
        return L.nrrt_accum_denoise(p._h, A.DenoiseOpts(**kw), ptr, 0)

    with gpu_ctx.progressive(cam) as p:  # plain handle: guides yes, filter no
        p.render(spp)
        p.aov()
        assert rc(p) == A.ERR_INVALID
    with gpu_ctx.progressive(cam, adaptive={"rel_error": 0.0}) as p:
        assert rc(p) == A.ERR_INVALID  # before the first pass
        p.aov(spp)                     # guides work before the first pass
        with pytest.raises(api.NrrtError):
            p.aov(spp + 1)
        p.render(spp)
        assert rc(p) == A.OK
        assert L.nrrt_accum_denoise(p._h, None, ptr, A.RENDER_OUT_PACKED) == A.ERR_INVALID
        assert L.nrrt_accum_denoise(p._h, None, ptr, 0) == A.OK
        for bad in ({"iterations": 9}, {"aov_samples": spp + 1}, {"sigma_color": -1.0}, {"sigma_color": float("inf")},
                    {"sigma_color": float("nan")}):
            assert rc(p, **bad) == A.ERR_INVALID, bad
    with gpu_ctx.progressive(cam, world=2, adaptive={"rel_error": 0.0}) as p:
        p.render(spp)
        assert rc(p) == A.ERR_INVALID
    with gpu_ctx.progressive(cam, adaptive={"rel_error": 0.0}) as p:
        p.render(spp)
        gpu_ctx.upload(hs)  # a replaced scene
        assert rc(p) == A.ERR_NO_SCENE
        assert L.nrrt_accum_aov(p._h, 0, ptr, None, 0) == A.ERR_NO_SCENE
    del hs


# Denoised RMSE over noisy RMSE after 64 spp, against a 4096-spp render of the same scene at 400x225: the largest ratio
# each scene may reach.  Measured (tools/denoise_time.py, DESIGN §4): Cornell 0.628, earth 0.322, teapot 0.534.
QUALITY = {"scenes/cornell-box-scene.json": 0.75, "scenes/earth.toml": 0.45, "scenes/utah-teapot-scene.json": 0.65}


@pytest.mark.parametrize("path", list(QUALITY))
def test_denoising_lowers_the_error(gpu_ctx, path):
    from tools.denoise_time import quality_rows
    [(spp, noisy, smooth)] = quality_rows(gpu_ctx, path, spps=[64])
    print(f"{path}: noisy {noisy:.5f} denoised {smooth:.5f} ratio {smooth / noisy:.3f}")
    assert smooth < noisy * QUALITY[path], (noisy, smooth)


def _png_pixels(path):
    """RGB8 pixels of a PNG with one IDAT and filter 0 rows (what the CLI writes)."""
    data = open(path, "rb").read()
    w, h = struct.unpack(">II", data[16:24])
    i, idat = 8, b""
    while i < len(data):
        n = struct.unpack(">I", data[i:i + 4])[0]
        if data[i + 4:i + 8] == b"IDAT":
            idat += data[i + 8:i + 8 + n]
        i += 12 + n
    raw = zlib.decompress(idat)
    rows = np.frombuffer(raw, np.uint8).reshape(h, 1 + 3 * w)
    assert (rows[:, 0] == 0).all()
    return rows[:, 1:].reshape(h, w, 3)


def test_cli_denoise(gpu_ctx, tmp_path):
    from nr_ray_tracer_b200 import build as B
    from nr_ray_tracer_b200.scene_config import CameraConfig
    B.build()
    W, H, spp = 96, 54, 40
    base = [B.CLI, "render", "scenes/cornell-box-scene.json", "-W", str(W), "-H", str(H), "--samples-per-pixel",
            str(spp), "--seed", "5"]
    out, prev = tmp_path / "d.png", tmp_path / "p.png"
    r = subprocess.run(base + ["-o", str(out), "--denoise"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    sc = api.Scene.load(os.path.join(ROOT, "scenes", "cornell-box-scene.json"), ctx=gpu_ctx,
                        camera_override=CameraConfig(width=W, height=H, samples_per_pixel=spp))
    image, den = sc.render_denoised(seed=5)
    assert np.array_equal(_png_pixels(out), gpu_ctx.encode_rgb8(den))
    r = subprocess.run(base + ["-o", str(prev), "--denoise", "--preview-every", "10"], capture_output=True, text=True,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert prev.read_bytes() == out.read_bytes()
    tol = tmp_path / "t.png"
    r = subprocess.run(base + ["-o", str(tol), "--denoise", "--adaptive-error", "0.05"], capture_output=True, text=True,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr
    _, den_t = sc.render_denoised(rel_error=0.05, seed=5)
    assert np.array_equal(_png_pixels(tol), gpu_ctx.encode_rgb8(den_t))
