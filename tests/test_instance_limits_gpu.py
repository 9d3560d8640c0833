"""Every render kernel and the fixed-ray query against the CPU oracle at the instance limits: nesting depth 4 (the
pooled kernel's packed chain words in full, and its rebuild of a parent level's ray when it leaves an instance), equal-t
ties whose instance chains first differ below level 0, instance ids past 16 bits (65536 instances, the pooled
kernel's limit, and 65537, which falls back to the fused kernel), and traversal stacks full by construction.

Bar for renders: every pixel bit-equal to the oracle's render summed in the kernels' work-item order, identical segment
and path counts, all designs identical.  On these scenes nothing transcendental runs on the device that could round
differently from libm: rotations are built on the host, the textures are a checker on quads (barycentric uv) and noise
(Perlin lattice arithmetic)."""
import numpy as np
import pytest

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200 import api
from oracle import oracle as O
from tools import instance_scenes as S
from tests import kat

pytestmark = pytest.mark.gpu
POOL_MIN_NODES = 1024   # NRRT_POOL_MIN_NODES: MODE_AUTO's pooled kernel from this many binary nodes


def _world_rays(hs, n, seed):
    """Rays from outside the scene's world box (root_box: wrappers applied) towards random points inside it."""
    rng = np.random.default_rng(seed)
    lo, hi = np.array(hs.desc.root_box.lo), np.array(hs.desc.root_box.hi)
    c, h = (lo + hi) / 2, (hi - lo) / 2
    target = c + (rng.random((n, 3)) * 2 - 1) * h
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = target - d * (np.linalg.norm(h) * rng.uniform(1.0, 2.0, size=(n, 1)))
    return np.concatenate([o, target - o], axis=1)


def _fixed_rays(ctx, g, hs, rays, levels=None):
    """kat bar against the oracle for both traversal modes; the chain the GPU reports is well formed: depth is a level
    at which the hit primitive occurs, ids below it index real instances, the compact output agrees.  Returns the hits."""
    import torch
    ref, _ = O.OracleScene(g).trace_rays(rays)
    d_rays = torch.from_numpy(np.ascontiguousarray(rays)).cuda()
    for visit_all in (False, True):
        gpu, _ = ctx.trace_rays(rays, visit_all=visit_all)
        res = kat.compare_hits(gpu, ref)
        assert kat.hits_ok(res), (visit_all, res)
        hit = gpu["object"] != 0xFFFFFFFF
        depth, inst = gpu["depth"][hit], gpu["inst"][hit]
        assert (depth <= A.MAX_INSTANCE_DEPTH).all()
        for l in range(A.MAX_INSTANCE_DEPTH):
            assert (inst[depth > l, l] < hs.desc.n_instances).all(), l
        if levels is not None:
            bad = [(int(o), int(dp)) for o, dp in zip(gpu["object"][hit], depth) if int(dp) not in levels[int(o)]]
            assert not bad, bad[:10]
        out = torch.zeros((len(rays), 16), dtype=torch.uint8, device="cuda")
        ctx.trace_rays_device(d_rays.data_ptr(), len(rays), out.data_ptr(), compact=True, visit_all=visit_all)
        torch.cuda.synchronize()
        c = out.cpu().numpy().view(np.dtype([("t", "<f8"), ("prim", "<u4"), ("depth_inst0", "<u4")])).reshape(-1)
        assert np.array_equal(c["depth_inst0"] & 7, gpu["depth"]) and np.array_equal(c["t"], gpu["t"])
    return gpu


def _designs(hs):
    out = [("wavefront", A.MODE_WAVEFRONT, None), ("megakernel", A.MODE_MEGAKERNEL, None), ("fused", A.MODE_FUSED, None),
           ("pool", A.MODE_POOL, "0")]
    if hs.desc.n_nodes < 64:   # the LITE pool variant walks the binary nodes, uploaded below 64 of them
        out.append(("pool-lite", A.MODE_POOL, "1"))
    return out + [("auto", A.MODE_AUTO, None)]


def _render_every_design(ctx, monkeypatch, g, hs, seed, auto_mode=None, fused_only=False):
    """Renders g in every kernel design and compares each with the oracle bit for bit.  Returns the image."""
    W, H, spp = g.camera.width, g.camera.height, g.camera.samples_per_pixel
    cam = api.camera_build(g.camera.to_builder_config())
    ref, cnt = O.OracleScene(g).render_chunked(O.camera_build(g.camera.to_builder_config()), api.chunk_starts(spp, W * H),
                                               seed=seed)
    assert cnt["paths"] == W * H * spp
    if auto_mode is None:
        auto_mode = A.MODE_POOL if hs.desc.n_nodes >= POOL_MIN_NODES else A.MODE_FUSED
    for label, mode, lite in _designs(hs):
        if lite is None:
            monkeypatch.delenv("NRRT_POOL_LITE", raising=False)
        else:
            monkeypatch.setenv("NRRT_POOL_LITE", lite)   # read by the library at render time
        img, st = ctx.render(cam, seed=seed, mode=mode)
        want_mode = {A.MODE_AUTO: auto_mode, A.MODE_POOL: A.MODE_FUSED if fused_only else A.MODE_POOL}.get(mode, mode)
        assert st["mode"] == want_mode, (label, st["mode"])
        diff = np.argwhere((img != ref).any(axis=2))
        assert len(diff) == 0, (label, len(diff), [(int(y), int(x), img[y, x].tolist(), ref[y, x].tolist())
                                                   for y, x in diff[:4]])
        assert (st["segments"], st["paths"]) == (cnt["segments"], cnt["paths"]), label
    monkeypatch.delenv("NRRT_POOL_LITE", raising=False)
    return ref


NESTED = [(d, o) for d in range(1, 5) for o in ("plain", "spec", "pool", "textured", "motion") if o != "motion" or d >= 3]
_KW = {"spec": {"mesh": "spec"}, "pool": {"mesh": "pool"}, "textured": {"textured": True}, "motion": {"motion": True}}


@pytest.mark.parametrize("depth,opt", [(d, o) for d, o in NESTED if o in ("plain", "spec", "pool")])
def test_fixed_rays_nested_instances(gpu_ctx, depth, opt):
    g, levels = S.nested(depth, **_KW.get(opt, {}))
    for bvh in ("reference", "sah"):
        hs = api.HostScene(g, bvh=bvh)
        gpu_ctx.upload(hs)
        rays = np.concatenate([_world_rays(hs, 40000, 3), kat.random_rays(g, 20000), kat.aimed_rays(g, 20000),
                               kat.special_rays(g)])
        gpu = _fixed_rays(gpu_ctx, g, hs, rays, levels)
        hit = gpu["object"] != 0xFFFFFFFF
        assert hit.sum() > 10000
        assert gpu["depth"][hit].max() == depth, (bvh, np.bincount(gpu["depth"][hit]))
        del hs


@pytest.mark.parametrize("depth,opt", NESTED)
def test_renders_nested_instances_in_every_design(gpu_ctx, monkeypatch, depth, opt):
    g, _ = S.nested(depth, **_KW.get(opt, {}))
    hs = api.HostScene(g)
    gpu_ctx.upload(hs)
    assert bool(hs.desc.sphere_speed) == (opt == "motion")
    _render_every_design(gpu_ctx, monkeypatch, g, hs, seed=17 + depth)
    del hs


@pytest.mark.parametrize("split", [2, 3])
def test_ties_between_chains_that_part_below_level_0(gpu_ctx, monkeypatch, split):
    g, pairs = S.coincident_across_levels(split)
    hs = api.HostScene(g)
    gpu_ctx.upload(hs)
    rays = np.concatenate([_world_rays(hs, 60000, 5), kat.aimed_rays(g, 60000, seed=8)])
    gpu = _fixed_rays(gpu_ctx, g, hs, rays)
    won = np.isin(gpu["object"], pairs["later"])
    assert won.sum() > 500 and not np.isin(gpu["object"], pairs["first"]).any()
    assert (gpu["depth"][won] == split + 1).all()
    img = _render_every_design(gpu_ctx, monkeypatch, g, hs, seed=9)
    # teeth: without the later pair the oracle's image is another one
    g0, _ = S.coincident_across_levels(split, with_later=False)
    alone, _ = O.OracleScene(g0).render_chunked(O.camera_build(g0.camera.to_builder_config()),
                                                api.chunk_starts(g0.camera.samples_per_pixel,
                                                                 g0.camera.width * g0.camera.height), seed=9)
    assert (alone != img).any(axis=2).mean() > 0.01
    del hs


@pytest.mark.parametrize("n_inner,level", [(65535, 1), (65534, 2)])
def test_65536_instances_ids_past_16_bits(gpu_ctx, monkeypatch, n_inner, level):
    """n_instances == 65536: the pooled kernel's limit.  The fan's ids reach 65533 / 65534 at `level` (the high half
    of the first packed word at level 1, the second word at level 2); the wrappers above it hold 65535 at level 0."""
    g = S.many_instances(n_inner, level)
    hs = api.HostScene(g)
    assert hs.desc.n_instances == 65536
    gpu_ctx.upload(hs)
    gpu = _fixed_rays(gpu_ctx, g, hs, np.concatenate([_world_rays(hs, 200000, 6), kat.aimed_rays(g, 50000)]))
    deep = (gpu["object"] != 0xFFFFFFFF) & (gpu["depth"] == level + 1)
    ids = gpu["inst"][deep, level]
    assert (ids >= 32768).sum() > 1000 and ids.max() >= 60000
    assert (gpu["inst"][deep, 0] == 65535).all()
    if level == 2:
        assert (gpu["inst"][deep, 1] == 65534).all()
    _render_every_design(gpu_ctx, monkeypatch, g, hs, seed=4)
    del hs


def test_65537_instances_fall_back_to_the_fused_kernel(gpu_ctx, monkeypatch):
    g = S.many_instances(65536, 1)
    hs = api.HostScene(g)
    assert hs.desc.n_instances == 65537 and hs.desc.n_nodes >= POOL_MIN_NODES
    gpu_ctx.upload(hs)
    _render_every_design(gpu_ctx, monkeypatch, g, hs, seed=4, auto_mode=A.MODE_FUSED, fused_only=True)
    del hs


@pytest.mark.parametrize("which", ["28", "32", "lite"])
def test_full_stacks_render_in_every_design(gpu_ctx, monkeypatch, which):
    g = S.lite_full_stack() if which == "lite" else S.full_stack(int(which))
    hs = api.HostScene(g)
    if which == "lite":
        assert hs.desc.n_nodes < 64 and S.binary_stack(hs) == 24
    else:
        assert hs.desc.max_stack == int(which)
    gpu_ctx.upload(hs)
    _fixed_rays(gpu_ctx, g, hs, np.concatenate([_world_rays(hs, 40000, 7), kat.aimed_rays(g, 20000)]))
    _render_every_design(gpu_ctx, monkeypatch, g, hs, seed=2)
    del hs


def test_scene_past_the_stack_cap_is_refused_at_upload(gpu_ctx):
    hs = api.HostScene(S.full_stack(33))
    assert hs.desc.max_stack == 33
    with pytest.raises(api.NrrtError) as e:
        gpu_ctx.upload(hs)
    assert e.value.code == A.ERR_LIMIT and "stack" in str(e.value)
