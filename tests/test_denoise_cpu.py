"""Denoising on the host side: properties of the filter's numpy statement (tests/denoise_ref.py) that follow from its
formula, a hand-derived case of the oracle's guides, the CLI's refusal of --denoise on several GPUs, and the ABI size of
nrrt_denoise_opts."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200 import api
from nr_ray_tracer_b200.scene_config import CameraConfig, SceneGraph
from oracle import oracle as O
from tests import aov_ref as AR
from tests import denoise_ref as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "nr_ray_tracer_b200", "bin", "nr-ray-tracer")
F = np.float32


def _random_inputs(H, W, seed, finite=True):
    rng = np.random.default_rng(seed)
    C_ = rng.random((H, W, 3)).astype(F) * F(3)
    e2 = (rng.random((H, W, 3)) * 0.05).astype(F)
    if not finite:
        e2[rng.random((H, W)) < 0.3] = np.inf
    albedo = rng.random((H, W, 3)).astype(F)
    albedo[rng.random((H, W)) < 0.2] = 0  # below the floor: demodulated by 2^-8
    n = rng.normal(size=(H, W, 3))
    normal = (n / np.linalg.norm(n, axis=-1, keepdims=True)).astype(F)
    normal[rng.random((H, W)) < 0.1] = 0  # misses
    return C_, e2, albedo, normal


def _scalar_denoise(C_, e2, albedo, normal, iterations, sigma_color):
    """The filter one pixel and one tap at a time with f32 scalars: every tap outside the image explicitly skipped."""
    H, W = C_.shape[:2]
    a = np.fmax(albedo, D.MIN_ALBEDO)
    E = C_ / a
    t = e2 / (a * a)
    v = ((t[..., 0] + t[..., 1]) + t[..., 2]) * (F(1) / F(9))
    s2 = F(sigma_color) * F(sigma_color)
    luma = lambda e: ((e[0] + e[1]) + e[2]) / F(3)
    dot = lambda p, q: (p[0] * q[0] + p[1] * q[1]) + p[2] * q[2]
    for it in range(iterations):
        h = 1 << it
        En, vn = np.zeros_like(E), np.zeros_like(v)
        for y in range(H):
            for x in range(W):
                lp, den = luma(E[y, x]), s2 * v[y, x] + D.EPS
                sw, sE, sv = F(0), np.zeros(3, F), F(0)
                for dy in range(-2, 3):
                    for dx in range(-2, 3):
                        qy, qx = y + dy * h, x + dx * h
                        if not (0 <= qy < H and 0 <= qx < W):
                            continue
                        w = D.B[abs(dx)] * D.B[abs(dy)]
                        if dx or dy:
                            wn = np.fmax(dot(normal[y, x], normal[qy, qx]), F(0))
                            for _ in range(7):
                                wn = wn * wn
                            d = albedo[y, x] - albedo[qy, qx]
                            wa = F(1) / (F(1) + dot(d, d) * F(64))
                            wc = F(1)
                            if v[y, x] != np.inf:
                                dl = lp - luma(E[qy, qx])
                                wc = F(1) / (F(1) + (dl * dl) / den)
                            w = ((w * wn) * wa) * wc
                        if w * w == 0:
                            continue
                        sw = sw + w
                        sE = sE + w * E[qy, qx]
                        sv = sv + (w * w) * v[qy, qx]
                En[y, x] = sE / sw
                vn[y, x] = sv / (sw * sw)
        E, v = En, vn
    return E * a


@pytest.mark.parametrize("H,W", [(1, 1), (1, 9), (9, 1), (2, 7), (6, 5), (9, 10)])
@pytest.mark.parametrize("finite", [True, False])
def test_vectorised_statement_skips_every_out_of_image_tap(H, W, finite):
    """At 1x1, 1xN, Nx1 and every border of small images (tap spacings up to 4, so most taps fall outside), the
    vectorised statement equals a per-pixel loop that skips each outside tap explicitly, bit for bit."""
    args = _random_inputs(H, W, H * 100 + W, finite)
    with np.errstate(all="ignore"):
        for iterations in (1, 3):
            ref = _scalar_denoise(*args, iterations, 4.0)
            out = D.denoise(*args, iterations=iterations)
            assert out.dtype == np.float32 and np.array_equal(out, ref), (iterations,)
            assert np.isfinite(out).all()


def test_single_pixel_keeps_its_value():
    C_, e2, albedo, normal = _random_inputs(1, 1, 3)
    out = D.denoise(C_, e2, albedo, normal, iterations=8)
    assert np.allclose(out, C_, rtol=2e-7, atol=0)


def test_pixel_whose_taps_all_fail_the_guides_keeps_its_value():
    """Normals facing away from the centre's (wn = 0) leave the centre tap alone: the pixel keeps C to rounding while its
    neighbours are smoothed."""
    H, W = 9, 9
    C_, e2, albedo, normal = _random_inputs(H, W, 5)
    normal[:] = (0, 0, 1)
    normal[4, 4] = (0, 0, -1)
    for it in (1, 5, 8):
        out = D.denoise(C_, e2, albedo, normal, iterations=it)
        assert np.allclose(out[4, 4], C_[4, 4], rtol=3e-7, atol=0), it
        assert not np.allclose(out[2, 2], C_[2, 2], rtol=1e-3)
    # the same for albedo: a centre whose albedo is far from all its neighbours' keeps a weight ratio of at least 1e3
    normal[4, 4] = (0, 0, 1)
    albedo[:] = 0.01
    albedo[4, 4] = 100.0
    out = D.denoise(C_, e2, albedo, normal, iterations=1)
    assert np.allclose(out[4, 4], C_[4, 4], rtol=1e-2, atol=0)


def test_no_error_estimate_gives_colour_weight_one_and_no_nan():
    """K < 2 everywhere: v = +inf, so wc = 1 (the result does not depend on sigma_color) and nothing is NaN."""
    H, W = 17, 33
    S = np.random.default_rng(1).random((H, W, 3)) * 40
    Q = S * S / 20  # any values: K < 2 ignores them
    N = np.full((H, W), 20)
    K = np.ones((H, W), int)
    C_, e2 = D.inputs(S, Q, N, K)
    assert np.isinf(e2).all()
    _, _, albedo, normal = _random_inputs(H, W, 2)
    a = D.denoise(C_, e2, albedo, normal, sigma_color=4.0)
    b = D.denoise(C_, e2, albedo, normal, sigma_color=0.001)
    assert np.array_equal(a, b) and np.isfinite(a).all()


def test_constant_image_stays_constant():
    H, W = 13, 21
    C_ = np.full((H, W, 3), F(0.3))
    e2 = np.full((H, W, 3), F(1e-3))
    albedo = np.full((H, W, 3), F(0.5))
    normal = np.zeros((H, W, 3), F)
    normal[..., 2] = 1
    out = D.denoise(C_, e2, albedo, normal, iterations=8)
    assert np.allclose(out, 0.3, rtol=1e-6, atol=0)


def _aov_graph():
    """A camera at (0, 0, 1) looking down -z with a 90 degree field of view sees [-1, 1]^2 at z = 0 as 8 x 8 pixels of
    0.25.  A Lambertian quad covers [-0.5, 0.5]^2 (pixel columns and rows 2..5), a light the top-right 2 x 2 pixels, a
    dielectric the bottom-left 2 x 2; the rest is background.  Colours are dyadic, so every mean is exact."""
    g = SceneGraph()
    lam = g.add_material(A.MAT_LAMBERTIAN, g.add_texture(kind=A.TEX_SOLID, color=(0.25, 0.5, 0.75)))
    light = g.add_material(A.MAT_DIFFUSE_LIGHT, g.add_texture(kind=A.TEX_SOLID, color=(4.0, 0.5, -2.0)), 3.0)
    glass = g.add_material(A.MAT_DIELECTRIC, 0, 1.5)
    q0 = g.add_object(A.OBJ_QUAD, lam, v=(-0.5, -0.5, 0, 1, 0, 0, 0, 1, 0))
    q1 = g.add_object(A.OBJ_QUAD, light, v=(0.5, 0.5, 0, 0.5, 0, 0, 0, 0.5, 0))
    q2 = g.add_object(A.OBJ_QUAD, glass, v=(-1.0, -1.0, 0, 0.5, 0, 0, 0, 0.5, 0))
    g.root = g.add_object(A.OBJ_GROUP, children=[q0, q1, q2])
    g.camera = CameraConfig(width=8, height=8, look_from=(0, 0, 1), look_at=(0, 0, 0), view_up=(0, 1, 0),
                            field_of_view=90.0, samples_per_pixel=4, background_color=(0.5, 2.0, -1.0))
    return g


def test_oracle_aov_hand_derived():
    g = _aov_graph()
    cam = O.camera_build(g.camera.to_builder_config())
    for n in (1, 4):
        albedo, normal = AR.oracle_aov(g, cam, n, seed=3)
        want_a = np.zeros((8, 8, 3), F)
        want_n = np.zeros((8, 8, 3), F)
        want_a[:] = (0.5, 1.0, 0.0)          # background, clamped
        want_a[2:6, 2:6] = (0.25, 0.5, 0.75)  # Lambertian: its texture colour
        want_a[0:2, 6:8] = (1.0, 0.5, 0.0)    # light: its colour clamped (row 0 is the top of the image)
        want_a[6:8, 0:2] = (1.0, 1.0, 1.0)    # dielectric
        want_n[2:6, 2:6] = want_n[0:2, 6:8] = want_n[6:8, 0:2] = (0, 0, 1)  # facing the camera; misses stay zero
        assert np.array_equal(albedo, want_a), n
        assert np.array_equal(normal, want_n), n
    # a pixel half on the quad: the mean of the hits' and misses' values over the first n samples
    g.camera.look_at = (0.125, 0.0, 0.0)
    g.camera.look_from = (0.125, 0.0, 1.0)  # shifts the view by half a pixel: columns 1 and 5 straddle the quad's edges
    cam = O.camera_build(g.camera.to_builder_config())
    albedo, normal = AR.oracle_aov(g, cam, 4, seed=3)
    frac = normal[2:6, 1, 2]  # the share of each pixel's samples that hit the quad
    assert ((frac * 4) % 1 == 0).all() and ((0 < frac) & (frac < 1)).any()
    assert (normal[2:6, 1, :2] == 0).all()
    want = frac[:, None] * np.array([0.25, 0.5, 0.75]) + (1 - frac[:, None]) * np.array([0.5, 1.0, 0.0])
    assert np.array_equal(albedo[2:6, 1], want.astype(F))


def test_cli_refuses_denoise_on_several_gpus(tmp_path):
    out = tmp_path / "d.png"
    r = subprocess.run([CLI, "render", os.path.join(ROOT, "scenes", "quads.toml"), "--denoise", "--gpus", "2", "-o",
                        str(out)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "--denoise renders on one GPU" in r.stderr
    assert not out.exists()
    r = subprocess.run([CLI, "render", "--help"], capture_output=True, text=True, timeout=60)
    assert "--denoise" in r.stdout


def test_denoise_opts_abi_size():
    L = api.lib()
    assert L.nrrt_abi_sizeof(20) == C.sizeof(A.DenoiseOpts) == 16
