"""Scene generators at the instance limits, for the tests and tools/sanitize_run.py: nesting depth up to
NRRT_MAX_INSTANCE_DEPTH (4), instance ids past 16 bits, traversal stacks filled to NRRT_STACK_CAP, and equal-t ties
whose instance chains first differ below level 0.

Plain functions returning a SceneGraph with a camera.  Wrapper chains (Translate / Rotate / Scale) become instances on
the host; a group with one child forwards to it, so every group here that must open a new instance level holds at
least two children."""
from __future__ import annotations

import math

import numpy as np

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200.scene_config import CameraConfig, SceneGraph

_WRAP = {"T": A.OBJ_TRANSLATE, "RX": A.OBJ_ROTATE_X, "RY": A.OBJ_ROTATE_Y, "RZ": A.OBJ_ROTATE_Z, "S": A.OBJ_SCALE}


def wrap(g: SceneGraph, chain, inner: int) -> int:
    """chain: [(kind, values), ...] outermost first."""
    for kind, v in reversed(chain):
        inner = g.add_object(_WRAP[kind], children=[inner], v=v if isinstance(v, tuple) else (v,))
    return inner


def _camera(g, width, height, spp, bounces, look_from=(0.0, 2.5, 11.0), fov=45.0):
    g.camera = CameraConfig(width=width, height=height, samples_per_pixel=spp, ray_max_bounces=bounces,
                            look_from=look_from, look_at=(0.0, 0.0, 0.0), background_color=(0.5, 0.7, 1.0),
                            field_of_view=fov)


def _height_field(g, mat, nx, nz, y0=-1.0, size=2.0):
    """2 nx nz triangles over a square of the given size: a mesh that makes a space's tree deep."""
    xs, zs = np.linspace(-size / 2, size / 2, nx + 1), np.linspace(-size / 2, size / 2, nz + 1)
    h = lambda x, z: y0 + 0.15 * math.sin(2.3 * x) * math.cos(1.9 * z)   # noqa: E731
    tris = []
    for i in range(nx):
        for j in range(nz):
            x0, x1, z0, z1 = xs[i], xs[i + 1], zs[j], zs[j + 1]
            p00, p10, p01, p11 = (x0, h(x0, z0), z0), (x1, h(x1, z0), z0), (x0, h(x0, z1), z1), (x1, h(x1, z1), z1)
            for a, b, c in ((p00, p10, p01), (p11, p01, p10)):
                tris.append(g.add_object(A.OBJ_TRIANGLE, mat, v=(*a, *np.subtract(b, a), *np.subtract(c, a))))
    return tris


# Wrapper chains of the fan instances, by fan index: every wrapper kind, non-uniform Scale included.
def _chain(level: int, j: int, fan: int):
    ang = 2.0 * math.pi * j / fan + 0.35 * level
    off = (1.9 * math.cos(ang), 0.35 * (j - 1), 1.9 * math.sin(ang))
    a = 0.3 + 0.41 * j + 0.17 * level
    return [[("T", off), ("RY", a), ("S", (0.6, 0.6, 0.6))],
            [("T", off), ("RX", a), ("S", (0.7, 0.5, 0.6))],
            [("T", off), ("RZ", -a), ("S", (0.55, 0.65, 0.5)), ("RY", 0.5 * a)]][j % 3]


def nested(depth: int, fan: int = 3, mesh: str = "", motion: bool = False, textured: bool = False, width: int = 64,
           height: int = 36, spp: int = 4, bounces: int = 8):
    """Instances nested `depth` levels deep (0..4).  The group at level k holds its own primitives next to `fan`
    wrapper chains around the group of level k + 1; the innermost group (a glass sphere, a quad, a light) is also
    wrapped directly from levels 1..depth-2, so its space is shared by instances at several levels.
      mesh: "" | "spec": a mesh in the innermost group (>= 64 binary nodes: the speculative fused kernel) |
            "pool": a larger mesh behind its own wrapper at level 0 (>= 1024 nodes: MODE_AUTO's pooled kernel; its
            tree in the innermost group would push the four levels' stack need past NRRT_STACK_CAP)
      motion: moving spheres in the level-3 group (NRRT_F_MOTION kernels): the innermost one at depth 3
      textured: checker texture on the quads, noise on level spheres
    Returns (graph, levels): levels[object id] = the set of nesting levels at which that primitive occurs."""
    assert 0 <= depth <= A.MAX_INSTANCE_DEPTH and (not motion or depth >= 3)
    g = SceneGraph()
    solid = [g.add_texture(kind=A.TEX_SOLID, color=c) for c in
             ((0.8, 0.3, 0.3), (0.3, 0.8, 0.4), (0.35, 0.4, 0.85), (0.9, 0.85, 0.6), (1.0, 1.0, 1.0))]
    if textured:
        chk = g.add_texture(kind=A.TEX_CHECKER, a=solid[3], b=solid[2], f0=6.0)
        noise = g.add_texture(kind=A.TEX_NOISE, seed=3, octaves=5, f0=1.3, f1=2.0, f2=0.5)
        quad_tex, ball_tex = chk, noise
    else:
        quad_tex, ball_tex = solid[3], solid[0]
    lam = g.add_material(A.MAT_LAMBERTIAN, ball_tex)
    lam2 = g.add_material(A.MAT_LAMBERTIAN, solid[1])
    lam_q = g.add_material(A.MAT_LAMBERTIAN, quad_tex)
    metal = g.add_material(A.MAT_METAL, solid[2], 0.25)
    glass = g.add_material(A.MAT_DIELECTRIC, 0, 1.5)
    light = g.add_material(A.MAT_DIFFUSE_LIGHT, solid[4], 3.0)
    levels = {}

    def prim(level, kind, mat, v):
        o = g.add_object(kind, mat, v=v)
        levels.setdefault(o, set()).add(level)
        return o

    core_prims = [(A.OBJ_SPHERE, glass, (0.0, 0.2, 0.0, 0.55)),
                  (A.OBJ_QUAD, lam_q, (-0.9, -0.6, -0.9, 1.8, 0, 0, 0, 0, 1.8)),
                  (A.OBJ_QUAD, light, (-0.3, 1.0, -0.3, 0.6, 0, 0, 0, 0, 0.6))]
    moving = [(A.OBJ_SPHERE, (lam, metal, glass)[i], (-1.0 + i, 1.6, 0.4, 0.3, 0.0, 0.4 * (i - 1), 0.3)) for i in range(3)]
    core_ids = [g.add_object(k, m, v=v) for k, m, v in core_prims + (moving if motion and depth == 3 else [])]
    if mesh == "spec":
        core_ids += _height_field(g, lam2, 4, 8)   # 64 triangles: depth 4 then needs 32 stack entries in both builds
    core = g.add_object(A.OBJ_GROUP, children=core_ids)
    for o in core_ids:
        levels[o] = {depth}
    inner = core
    for k in range(depth - 1, -1, -1):
        kids = [prim(k, A.OBJ_SPHERE, (lam, metal, lam2)[k % 3], (0.0, -1.5, 0.0, 0.45)),
                prim(k, A.OBJ_TRIANGLE, lam2, (-2.2, -1.9, -1.5, 0.9, 0.0, 0.3, 0.1, 1.2, 0.0))]
        if motion and k == 3:
            kids += [prim(k, *m) for m in moving]
        kids += [wrap(g, _chain(k, j, fan), inner) for j in range(fan)]
        if 1 <= k <= depth - 2:   # the innermost space once more, directly from this level
            kids.append(wrap(g, [("T", (0.0, 2.1, -0.8)), ("S", (0.5, 0.5, 0.5))], core))
            for o in core_ids:
                levels[o].add(k + 1)
        inner = g.add_object(A.OBJ_GROUP, children=kids)
    if depth == 0:   # no instance at all: the innermost group is the scene
        inner = g.add_object(A.OBJ_GROUP, children=core_ids + [prim(0, A.OBJ_SPHERE, lam, (0.0, -1.5, 0.0, 0.45))])
    top = [inner, prim(0, A.OBJ_QUAD, lam_q, (-8.0, -2.6, -8.0, 16.0, 0, 0, 0, 0, 16.0))]
    if mesh == "pool":   # a space of its own: inside the innermost group its depth would add to the four levels'
        tris = _height_field(g, lam2, 24, 24, size=6.0)
        for o in tris:
            levels[o] = {1}
        top.append(wrap(g, [("T", (0.0, -0.5, -1.0)), ("RY", 0.25)], g.add_object(A.OBJ_GROUP, children=tris)))
    g.root = g.add_object(A.OBJ_GROUP, children=top)
    _camera(g, width, height, spp, bounces)
    return g, levels


def coincident_across_levels(split_level: int, with_later: bool = True, width: int = 48, height: int = 27, spp: int = 4):
    """Two different primitive pairs (a quad and a sphere each), with different object ids and materials, that
    coincide exactly in world space.  They sit behind instance chains whose ids agree above `split_level` (2 or 3) and
    differ there: the two instances at that level carry the same wrapper values (dyadic translations, power-of-two
    scales), so both sides compute bit-identical rays and every ray that hits one hits the other at the same t.  The
    reference keeps the later leaf (object.rs:110-114), which tie_candidate_wins finds by comparing the chains level by
    level.  with_later=False drops the later pair (a scene whose image must differ)."""
    assert split_level in (2, 3)
    g = SceneGraph()
    red = g.add_material(A.MAT_LAMBERTIAN, g.add_texture(kind=A.TEX_SOLID, color=(0.8, 0.2, 0.2)))
    green = g.add_material(A.MAT_METAL, g.add_texture(kind=A.TEX_SOLID, color=(0.2, 0.8, 0.3)), 0.125)
    grey = g.add_material(A.MAT_LAMBERTIAN, g.add_texture(kind=A.TEX_SOLID, color=(0.5, 0.5, 0.5)))
    lamp = g.add_material(A.MAT_DIFFUSE_LIGHT, g.add_texture(kind=A.TEX_SOLID, color=(1.0, 1.0, 1.0)), 2.0)

    def pair(mat):
        return [g.add_object(A.OBJ_QUAD, mat, v=(-1.0, -1.0, 0.0, 2.0, 0, 0, 0, 2.0, 0)),
                g.add_object(A.OBJ_SPHERE, mat, v=(0.5, 0.25, 0.5, 0.75))]
    first = pair(red)
    later = pair(green) if with_later else []
    split_chain = [("T", (0.25, -0.5, 0.125)), ("S", (2.0, 2.0, 2.0))]
    split = [wrap(g, split_chain, g.add_object(A.OBJ_GROUP, children=first))]
    if with_later:
        split.append(wrap(g, split_chain, g.add_object(A.OBJ_GROUP, children=later)))
    inner = g.add_object(A.OBJ_GROUP, children=split + [g.add_object(A.OBJ_SPHERE, grey, v=(6.0, 0.0, 0.0, 0.5))])
    for k in range(split_level - 1, -1, -1):   # one wrapper chain per level above the split, each around a group
        chain = [("T", (0.5 * k - 0.25, 0.25, -0.5)), ("S", (0.5, 0.5, 0.5))] if k % 2 else [("T", (0.0, 0.5, 0.25))]
        filler = g.add_object(A.OBJ_SPHERE, grey, v=(-6.0 - k, 1.0, 0.0, 0.5))
        inner = g.add_object(A.OBJ_GROUP, children=[wrap(g, chain, inner), filler])
    g.root = g.add_object(A.OBJ_GROUP, children=[inner, g.add_object(A.OBJ_QUAD, lamp, v=(-4.0, 5.0, -4.0, 8.0, 0, 0, 0, 0, 8.0)),
                                                 g.add_object(A.OBJ_QUAD, grey, v=(-8.0, -3.0, -8.0, 16.0, 0, 0, 0, 0, 16.0))])
    _camera(g, width, height, spp, 6, look_from=(0.5, 1.5, 6.0), fov=40.0)
    return g, {"first": first, "later": later}


def many_instances(n_inner: int, level: int = 1, width: int = 48, height: int = 27, spp: int = 2):
    """`n_inner` instances of one shared group (a sphere and a quad), each with its own rotation and translation, in a
    group nested `level` instance levels deep (1 or 2).  n_instances = n_inner + level.  The host numbers an instance
    after everything inside it, so the fan's ids are 0 .. n_inner - 1 and the wrappers above it take the last ids.
    (At level 3 a fan of more than 32768 instances needs a 34-entry stack: past NRRT_STACK_CAP.)"""
    assert level in (1, 2)
    g = SceneGraph()
    mats = [g.add_material(A.MAT_LAMBERTIAN, g.add_texture(kind=A.TEX_SOLID, color=c))
            for c in ((0.8, 0.4, 0.3), (0.3, 0.6, 0.8))]
    metal = g.add_material(A.MAT_METAL, g.add_texture(kind=A.TEX_SOLID, color=(0.8, 0.8, 0.7)), 0.1)
    shared = g.add_object(A.OBJ_GROUP, children=[g.add_object(A.OBJ_SPHERE, mats[0], v=(0.3, 0.0, 0.0, 0.35)),
                                                 g.add_object(A.OBJ_QUAD, mats[1], v=(-0.4, -0.4, 0.0, 0.8, 0, 0, 0, 0.5, 0))])
    side = int(math.ceil(math.sqrt(n_inner)))
    step = 8.0 / side
    kinds = ("RX", "RY", "RZ")
    fan = []
    for i in range(n_inner):
        x, z = -4.0 + step * (i % side + 0.5), -4.0 + step * (i // side + 0.5)
        fan.append(wrap(g, [("T", (x, 0.0, z)), ("S", (0.45 * step,) * 3), (kinds[i % 3], 0.1 + 6.1 * i / n_inner)],
                        shared))
    inner = g.add_object(A.OBJ_GROUP, children=fan)
    for k in range(level - 1, -1, -1):
        inner = g.add_object(A.OBJ_GROUP, children=[
            wrap(g, [("T", (0.0, 0.2 * k, 0.0)), ("RY", 0.2 + 0.1 * k)], inner),
            g.add_object(A.OBJ_SPHERE, metal, v=(5.5 + k, 0.5, 0.0, 0.5))])
    g.root = inner
    _camera(g, width, height, spp, 4, look_from=(0.0, 7.0, 7.0), fov=50.0)
    return g


def _stacked(counts, sizes=None):
    """Depth-4 nesting whose level-k group holds counts[k] primitives around one wrapper chain of the next level
    (counts has 5 entries; the last is the innermost group).  The primitives sit on a line sorted by x so the
    instance leaf lands where the reference's median split puts the last child."""
    g = SceneGraph()
    m = g.add_material(A.MAT_LAMBERTIAN, g.add_texture(kind=A.TEX_SOLID, color=(0.7, 0.6, 0.5)))
    lamp = g.add_material(A.MAT_DIFFUSE_LIGHT, g.add_texture(kind=A.TEX_SOLID, color=(1.0, 1.0, 1.0)), 2.0)
    inner = None
    for k in range(len(counts) - 1, -1, -1):
        n = counts[k]
        kids = [g.add_object(A.OBJ_SPHERE, lamp if (k + i) % 7 == 0 else m,
                             v=(-2.0 + 4.0 * i / max(n, 1), 0.3 * math.sin(i + k), -0.5 * k, 0.6 * 4.0 / max(n, 1)))
                for i in range(n)]
        if inner is not None:
            kids.append(wrap(g, [("T", (0.25, 0.125 * k, 0.5)), ("RY", 0.3 + 0.2 * k), ("S", (0.75, 0.5, 0.75))], inner))
        inner = g.add_object(A.OBJ_GROUP, children=kids)
    g.root = g.add_object(A.OBJ_GROUP, children=[inner, g.add_object(A.OBJ_QUAD, m, v=(-6.0, -1.5, -6.0, 12.0, 0, 0, 0, 0, 12.0))])
    _camera(g, 40, 24, 2, 6, look_from=(0.0, 2.0, 7.0), fov=50.0)
    return g


def binary_stack(hs) -> int:
    """Traversal stack entries over the BINARY nodes (what the LITE pool variant and the plain fused kernel walk):
    the upload's binary_stack_need + 2 (nrrt_device.cu)."""
    d = hs.desc
    nodes = hs.nodes()
    inst_inner = [d.instances[i].inner for i in range(d.n_instances)]
    memo = {}

    def below(ref):
        if ref == A.REF_NONE:
            return 0
        ty, ix = ref >> A.REF_TYPE_SHIFT, ref & A.REF_INDEX_MASK
        if ty == A.REF_NODE:
            if ref not in memo:
                memo[ref] = 1 + max(below(int(c)) for c in nodes["child"][ix])
            return memo[ref]
        if ty == A.REF_INSTANCE:
            return 1 + below(int(inst_inner[ix]))
        return 0
    return below(int(d.root)) + 2


# Per-level primitive counts, found by search over the host build and pinned here: the stack needs they give are
# asserted by the tests, so a change of the host build that moves them fails loudly instead of quietly testing less.
FULL_STACK_COUNTS = {28: (2, 2, 13, 13, 15), 32: (5, 5, 15, 15, 15), 33: (5, 5, 17, 17, 15)}
LITE_CAP_COUNTS = (8, 8, 13, 13, 8)   # binary stack 24 over 50 nodes (27 is the most any count gives under 64 nodes)


def full_stack(target: int):
    """Depth-4 scene whose host max_stack (four-slot nodes) is exactly `target` (28, 32, or 33 = one past the cap)."""
    return _stacked(FULL_STACK_COUNTS[target])


def lite_full_stack():
    """Depth-4 scene under 64 binary nodes whose binary stack need + 2 is 24, a multiple of 4: the LITE variant's
    per-scene cap with no rounding slack (28 is out of reach under 64 nodes at this nesting)."""
    return _stacked(LITE_CAP_COUNTS)


def instance_levels(hs):
    """{instance id: set of nesting levels at which it is entered}, walking the four-slot nodes from wide_root as the
    kernels do (level 0 = world space)."""
    wn, inner = hs.wnodes(), hs.instance_wide_inner()
    out, seen = {}, set()

    def walk(ref, level):
        if ref == A.REF_NONE or (ref, level) in seen:
            return
        seen.add((ref, level))
        ty, ix = ref >> A.REF_TYPE_SHIFT, ref & A.REF_INDEX_MASK
        if ty == A.REF_NODE:
            for c in wn["child"][ix]:
                walk(int(c), level)
        elif ty == A.REF_INSTANCE:
            out.setdefault(int(ix), set()).add(level)
            walk(int(inner[ix]), level + 1)
    walk(int(hs.desc.wide_root), 0)
    return out


def all_scenes():
    """{name: builder} of every generated scene small enough to walk in Python, for the layout checks."""
    out = {}
    for depth in range(5):
        for kw in ({}, {"mesh": "spec"}, {"mesh": "pool"}, {"textured": True}) + (({"motion": True},) if depth >= 3 else ()):
            out[f"nested{depth}" + "".join(f"-{k}={v}" for k, v in kw.items())] = \
                lambda depth=depth, kw=kw: nested(depth, **kw)[0]
    for s in (2, 3):
        out[f"coincident{s}"] = lambda s=s: coincident_across_levels(s)[0]
    for k in (28, 32):
        out[f"full_stack{k}"] = lambda k=k: full_stack(k)
    out["lite_full_stack"] = lite_full_stack
    return out
