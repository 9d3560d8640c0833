"""Adaptive sampling on the GPU (nrrt_accum_create_adaptive, Context.progressive(adaptive=...), Scene.render_adaptive,
--adaptive-error): with zero tolerance the frame is nrrt_render's image bit for bit; with a positive one every pixel is
the oracle's render over the chunks it received, its state is the chunk partials reduced in the stated order (and the
oracle's to rounding), the retired set is the numpy test on that state, and none of it depends on the kernel design,
slot count or partition."""
import os
import subprocess

import numpy as np
import pytest

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200 import api
from oracle import oracle as O
from tests import adaptive_ref as R
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


def _frame(ctx, cam, targets, adaptive, **kw):
    """Runs an adaptive frame to each target in turn (stopping once no pixel is active).  Returns a list of passes:
    dict(samples, active, stats, image, error, map, S, Q, N)."""
    out = []
    with ctx.progressive(cam, adaptive=adaptive, **kw) as p:
        assert p.active == p.rows * cam.width
        for t in targets:
            if not p.active:
                break
            st = p.render(t)
            S, Q, N = p.state()
            out.append(dict(samples=p.samples, active=p.active, stats=st, image=p.image(), error=p.error_image(),
                            map=p.sample_map(), S=S, Q=Q, N=N))
    return out


def _boundaries(starts):
    """Pass targets: one pass per chunk, [1 chunk, rest], doubling chunk counts."""
    n = len(starts) - 1
    dbl, k = [], 1
    while k < n:
        dbl.append(starts[k])
        k *= 2
    return {"per chunk": starts[1:], "[1, rest]": [starts[1], starts[-1]], "doubling": dbl + [starts[-1]]}


@pytest.mark.parametrize("name", SCENES)
def test_zero_tolerance_is_the_one_shot_render(gpu_ctx, name):
    W, H, spp = 64, 36, 40
    g, hs, cam = _setup(gpu_ctx, name, width=W, height=H, samples_per_pixel=spp, ray_max_bounces=10)
    starts = api.chunk_starts(spp, W * H)
    for mode in MODES:
        ref, st = gpu_ctx.render(cam, seed=9, mode=mode)
        for label, targets in _boundaries(starts).items():
            passes = _frame(gpu_ctx, cam, targets, {"rel_error": 0.0, "min_samples": 0}, seed=9, mode=mode)
            last = passes[-1]
            assert np.array_equal(last["image"], ref), (name, mode, label)
            assert last["samples"] == spp and last["active"] == 0 and (last["map"] == spp).all()
            assert all(p["active"] == W * H for p in passes[:-1])
            assert sum(p["stats"]["paths"] for p in passes) == st["paths"] == W * H * spp
            assert sum(p["stats"]["segments"] for p in passes) == st["segments"], (name, mode, label)
    del hs


def _gpu_partials(ctx, cam, starts, seed):
    """(H, W, n_chunks, 3) f64: each chunk's partial sums as the GPU computes them — a plain progressive frame restored
    to zero sums at chunk c's start and rendered through chunk c holds exactly 0 + P_c."""
    out = np.zeros((cam.height, cam.width, len(starts) - 1, 3))
    zero = np.zeros((cam.height, cam.width, 3))
    with ctx.progressive(cam, seed=seed) as p:
        for c in range(len(starts) - 1):
            p.restore(starts[c], zero)
            p.render(starts[c + 1])
            out[:, :, c] = p.state()[1]
    return out


def _check_exact(passes, cam, starts, partials, osc, ocam, tol, seed, oracle_partials):
    """Every pass of an adaptive frame against the chunk partials reduced in the stated order, the oracle and the numpy
    test.  The device's f64 partials agree with the oracle's to rounding: its sin / cos / atan2 / pow are not the host
    libm's, which an f32 image does not show but f64 sums can."""
    H, W = cam.height, cam.width
    spp = starts[-1]
    retired = np.zeros((H, W), bool)
    prev = None
    chunk_of = {s: k for k, s in enumerate(starts)}
    renders = {}
    for i, p in enumerate(passes):
        S, Q, N = p["S"], p["Q"], p["N"]
        K = np.vectorize(chunk_of.get)(N)
        S_ref, Q_ref = R.reduce_partials(partials, starts, K)
        assert np.array_equal(S, S_ref) and np.array_equal(Q, Q_ref), i
        S_or, Q_or = R.reduce_partials(oracle_partials, starts, K)
        assert np.allclose(S, S_or, rtol=1e-12, atol=1e-300) and np.allclose(Q, Q_or, rtol=1e-12, atol=1e-300), i
        assert np.array_equal(p["map"], N)
        conv = R.converged(S, Q, N, K, tol["rel_error"], tol.get("abs_error", 0.0), tol["min_samples"])
        boundary = N.max()
        assert boundary == p["samples"]
        # retired = passed the test, or below the boundary; a pixel below the boundary passed it at its last pass
        assert (conv[N < boundary]).all()
        now_retired = (N < boundary) | conv | (N == spp)
        assert p["active"] == int((~now_retired).sum()), i
        if prev is not None:  # a retired pixel's state never changes again
            for a, b in ((S, prev["S"]), (Q, prev["Q"]), (N, prev["N"])):
                assert np.array_equal(a[retired], b[retired]), i
            # the pass rendered exactly the pixels active before it
            ran = ~retired
            assert p["stats"]["pixels"] == int(ran.sum())
            assert (N[ran] == boundary).all()
            assert p["stats"]["paths"] == int(ran.sum()) * (boundary - prev["samples"])
        retired = now_retired
        # the image: each pixel the oracle's render_chunked over its own chunks
        want = np.empty((H, W, 3), np.float32)
        for k in np.unique(K):
            if k not in renders:
                renders[k], _ = osc.render_chunked(ocam, starts[:k + 1], seed=seed)
            want[K == k] = renders[k][K == k]
        assert np.array_equal(p["image"], want), i
        assert np.array_equal(p["image"], (S / N[..., None]).astype(np.float32))
        err = np.where((K >= 2)[..., None], np.sqrt(R.e2(S, Q, N, np.maximum(K, 2))), np.inf).astype(np.float32)
        assert np.array_equal(p["error"], err), i
        prev = p
    return retired


@pytest.mark.parametrize("name", ["spheres.toml", "earth.toml", "cornell-box-scene.json"])
def test_retirement_is_exact_against_the_oracle(gpu_ctx, name):
    W, H, spp, seed = 40, 24, 48, 6
    g, hs, cam = _setup(gpu_ctx, name, width=W, height=H, samples_per_pixel=spp, ray_max_bounces=50)
    starts = api.chunk_starts(spp, W * H)
    osc, ocam = O.OracleScene(g), O.camera_build(g.camera.to_builder_config())
    oracle_partials = R.render_partials(g, ocam, starts, seed=seed)
    partials = _gpu_partials(gpu_ctx, cam, starts, seed)
    found = False
    for rel in (0.01, 0.05, 0.002, 0.2):
        tol = {"rel_error": rel, "min_samples": starts[2]}
        passes = _frame(gpu_ctx, cam, [starts[2], starts[4], starts[8], starts[16], spp], tol, seed=seed)
        retired_early = passes[-1]["map"] < spp
        if retired_early.any() and not retired_early.all():
            _check_exact(passes, cam, starts, partials, osc, ocam, tol, seed, oracle_partials)
            found = True
            break
    assert found, name  # some tolerance retires some pixels early but not all
    del hs


def test_design_slots_and_partition_do_not_change_the_result(gpu_ctx):
    W, H, spp, seed = 48, 27, 40, 2
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=50)
    starts = api.chunk_starts(spp, W * H)
    tol = {"rel_error": 0.02, "abs_error": 1e-3, "min_samples": starts[2]}
    targets = [starts[2], starts[5], starts[10], spp]
    ref = _frame(gpu_ctx, cam, targets, tol, seed=seed, mode=A.MODE_FUSED)
    assert 0 < (ref[-1]["map"] < spp).sum() < W * H
    one_shot, st = gpu_ctx.render(cam, seed=seed, mode=A.MODE_FUSED)
    assert sum(p["stats"]["segments"] for p in ref) < st["segments"]
    full_pass = ref[-1]["map"] == spp
    assert np.array_equal(ref[-1]["image"][full_pass], one_shot[full_pass])
    keys = ("S", "Q", "N", "map", "image", "error")
    for mode in MODES:
        for max_slots in (0, 777):
            got = _frame(gpu_ctx, cam, targets, tol, seed=seed, mode=mode, max_slots=max_slots)
            assert len(got) == len(ref)
            for a, b in zip(got, ref):
                assert a["samples"] == b["samples"] and a["active"] == b["active"]
                assert a["stats"]["paths"] == b["stats"]["paths"]
                for k in keys:
                    assert np.array_equal(a[k], b[k]), (mode, max_slots, k)
    for world, rpb in ((2, 1), (3, 8)):
        S = np.full_like(ref[-1]["S"], np.nan)
        N = np.zeros_like(ref[-1]["N"])
        img = np.full_like(ref[-1]["image"], np.nan)
        for rank in range(world):
            rows = np.array([y for y in range(H) if (y // rpb) % world == rank], dtype=np.int64)
            with gpu_ctx.progressive(cam, seed=seed, rank=rank, world=world, rows_per_block=rpb, adaptive=tol) as p:
                for t in targets:
                    if p.active:
                        p.render(t)
                s, q, n = p.state()
                S[rows], N[rows] = s, n
                assert np.array_equal(q, ref[-1]["Q"][rows])
                assert np.array_equal(p.sample_map(packed=True), ref[-1]["N"][rows])
                assert np.array_equal(p.image(packed=True), ref[-1]["image"][rows])
                p.image(out=img)
        assert np.array_equal(S, ref[-1]["S"]) and np.array_equal(N, ref[-1]["N"]), world
        assert np.array_equal(img, ref[-1]["image"]), world
    del hs


def test_device_outputs(gpu_ctx):
    import torch
    W, H, spp = 32, 20, 16
    g, hs, cam = _setup(gpu_ctx, "spheres.toml", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=20)
    with gpu_ctx.progressive(cam, seed=1, adaptive={"rel_error": 0.05}) as p:
        assert (p.sample_map() == 0).all() and np.isinf(p.error_image()).all()
        p.render(spp // 2)
        d = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        p.sample_map(out_device_ptr=d.data_ptr())
        assert np.array_equal(d.cpu().numpy().view(np.uint32), p.sample_map())
        e = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda")
        p.error_image(out_device_ptr=e.data_ptr())
        assert np.array_equal(e.cpu().numpy(), p.error_image())
        i = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda")
        p.image(out_device_ptr=i.data_ptr())
        assert np.array_equal(i.cpu().numpy(), p.image())
    del hs


def test_resume_and_restore_validation(gpu_ctx):
    W, H, spp, seed = 48, 27, 40, 3
    g, hs, cam = _setup(gpu_ctx, "spheres.toml", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=30)
    starts = api.chunk_starts(spp, W * H)
    tol = {"rel_error": 0.03, "min_samples": starts[2]}
    targets = [starts[2], starts[4], starts[8], spp]
    ref = _frame(gpu_ctx, cam, targets, tol, seed=seed)
    assert 0 < (ref[-1]["map"] < spp).sum() < W * H
    with gpu_ctx.progressive(cam, seed=seed, adaptive=tol) as p:
        p.render(targets[0])
        p.render(targets[1])
        S, Q, N = p.state()
        active = p.active
    assert 0 < active < W * H
    ctx2 = api.Context(0)
    try:
        hs2 = api.HostScene(g)
        ctx2.upload(hs2)
        with ctx2.progressive(cam, seed=seed, adaptive=tol) as q:
            bad_n = N.copy()
            bad_n[3, 4] = starts[1] + 1  # not a chunk boundary
            with pytest.raises(api.NrrtError) as e:
                q.restore(S, Q, bad_n)
            assert e.value.code == A.ERR_INVALID
            # an active pixel moved below the boundary without passing the test
            act = np.argwhere(N == N.max())
            y, x = act[0]
            bad_n, bad_q = N.copy(), Q.copy()
            bad_n[y, x] = starts[1]
            bad_q[y, x] += 1e6
            with pytest.raises(api.NrrtError) as e:
                q.restore(S, bad_q, bad_n)
            assert e.value.code == A.ERR_INVALID
            # a fresh frame's state with something already summed
            dirty = np.zeros_like(S)
            dirty[1, 2, 0] = 0.5
            for bad_s, bad_q in ((dirty, np.zeros_like(Q)), (np.zeros_like(S), dirty)):
                with pytest.raises(api.NrrtError) as e:
                    q.restore(bad_s, bad_q, np.zeros_like(N))
                assert e.value.code == A.ERR_INVALID
            with pytest.raises(ValueError):
                q.restore(S[:-1], Q, N)
            with pytest.raises(ValueError):
                q.restore(S, Q, N.ravel()[:-2])
            q.restore(S, Q, N)
            assert q.active == active and q.samples == targets[1]
            for t in targets[2:]:
                if q.active:
                    q.render(t)
            S2, Q2, N2 = q.state()
            assert np.array_equal(S2, ref[-1]["S"]) and np.array_equal(Q2, ref[-1]["Q"])
            assert np.array_equal(N2, ref[-1]["N"]) and np.array_equal(q.image(), ref[-1]["image"])
            # a fresh frame's empty state restores to a fresh frame
            with ctx2.progressive(cam, seed=seed, adaptive=tol) as r:
                r.restore(np.zeros_like(S), np.zeros_like(Q), np.zeros_like(N))
                assert r.active == W * H and r.samples == 0
            ctx2.upload(hs2)  # replacing the scene invalidates the frame
            for call in (lambda: q.render(spp), q.image, q.state, q.sample_map, q.error_image,
                         lambda: q.restore(S, Q, N)):
                with pytest.raises(api.NrrtError) as e:
                    call()
                assert e.value.code == A.ERR_NO_SCENE
        del hs2
    finally:
        ctx2.close()
    del hs


def test_invalid_calls(gpu_ctx):
    import ctypes as C
    W, H, spp = 16, 9, 8
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=spp)
    for bad in ({"rel_error": -0.1}, {"rel_error": float("nan")}, {"rel_error": 0.1, "abs_error": float("inf")},
                {"rel_error": 0.1, "abs_error": -1.0}):
        with pytest.raises(api.NrrtError) as e:
            gpu_ctx.progressive(cam, adaptive=bad)
        assert e.value.code == A.ERR_INVALID
    with gpu_ctx.progressive(cam, adaptive={"rel_error": 0.1}) as p:
        p.render(spp)
        n = C.c_uint32()
        sums = np.zeros((H, W, 3))
        assert api.lib().nrrt_accum_save(p._h, C.c_void_p(sums.ctypes.data), C.byref(n)) == A.ERR_INVALID
        assert api.lib().nrrt_accum_restore(p._h, C.c_void_p(sums.ctypes.data), spp) == A.ERR_INVALID
    with gpu_ctx.progressive(cam) as p:
        p.render(spp)
        assert p.active == 0
        for call in (p.sample_map, p.error_image):
            with pytest.raises(api.NrrtError) as e:
                call()
            assert e.value.code == A.ERR_INVALID
        z = np.zeros((H, W, 3))
        zn = np.zeros((H, W), np.uint32)
        assert api.lib().nrrt_accum_adaptive_save(p._h, C.c_void_p(z.ctypes.data), C.c_void_p(z.ctypes.data),
                                                  C.c_void_p(zn.ctypes.data)) == A.ERR_INVALID
        assert api.lib().nrrt_accum_adaptive_restore(p._h, C.c_void_p(z.ctypes.data), C.c_void_p(z.ctypes.data),
                                                     C.c_void_p(zn.ctypes.data)) == A.ERR_INVALID
    del hs


def test_scene_render_adaptive(gpu_ctx):
    from nr_ray_tracer_b200.scene_config import CameraConfig
    s = api.Scene.load("scenes/spheres.toml", camera_override=CameraConfig(width=48, height=27, samples_per_pixel=64),
                       ctx=gpu_ctx)
    ref = s.render(seed=2)
    starts = api.chunk_starts(64, 48 * 27)
    got = list(s.render_adaptive(0.0, seed=2))
    ms = api.default_min_samples(64, 48 * 27)
    k0 = starts.index(ms)
    want, k = [], k0
    while k < len(starts) - 1:
        want.append(starts[k])
        k *= 2
    assert [n for n, _, _ in got] == want + [64]
    assert np.array_equal(got[-1][2], ref) and got[-1][1] == 0
    got = list(s.render_adaptive(0.05, every=16, seed=2))
    assert got[-1][1] == 0 and all(a > 0 for _, a, _ in got[:-1])


def test_benchmark_workload_with_a_tolerance(gpu_ctx):
    W, H, spp = 1920, 1080, 1024
    g, hs, cam = _setup(gpu_ctx, "cornell-box-scene.json", width=W, height=H, samples_per_pixel=spp, ray_max_bounces=50)
    ref, st = gpu_ctx.render(cam, seed=0, mode=A.MODE_AUTO)
    starts = api.chunk_starts(spp, W * H)
    segs = 0
    with gpu_ctx.progressive(cam, seed=0, adaptive={"rel_error": 0.03}) as p:
        k = starts.index(api.default_min_samples(spp, W * H))
        while p.active:
            segs += p.render(starts[min(k, len(starts) - 1)])["segments"]
            k *= 2
        N = p.sample_map()
        img = p.image()
    full = N == spp
    assert np.isin(N, starts[1:]).all()
    assert np.array_equal(img[full], ref[full])
    if not full.all():
        assert segs < st["segments"]
    del hs


def test_cli_adaptive(gpu_ctx, tmp_path):
    from nr_ray_tracer_b200 import build as B
    B.build()
    base = [B.CLI, "render", "scenes/cornell-box-scene.json", "-W", "96", "-H", "54", "--samples-per-pixel", "40",
            "--seed", "5"]
    plain, zero, tol = tmp_path / "plain.png", tmp_path / "zero.png", tmp_path / "tol.png"
    r = subprocess.run(base + ["-o", str(plain)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    r = subprocess.run(base + ["-o", str(zero), "--adaptive-error", "0"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert zero.read_bytes() == plain.read_bytes()
    r = subprocess.run(base + ["-o", str(tol), "--adaptive-error", "0.05", "--adaptive-abs-error", "0.001", "-v"],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert tol.exists() and tol.stat().st_size == plain.stat().st_size  # an uncompressed PNG of the same size
    lines = [line.split() for line in r.stderr.splitlines() if line.startswith("pass: ")]
    assert lines and all("active" in ln for ln in lines)
    active = [int(ln[ln.index("active") - 1]) for ln in lines]
    assert active[-1] == 0 and all(a > 0 for a in active[:-1])
    assert not [f for f in os.listdir(tmp_path) if ".tmp" in f]
