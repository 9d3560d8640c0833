"""CPU oracle checks: Philox known answers, hand-derivable intersection cases and the reference's quirks
(SURVEY.md §8 Q1-Q10, §4 level 1), and the committed golden fixtures.

The reference has no tests or golden vectors of its own and cannot be run here, so the hand-derived cases
below (each citing the reference lines that imply the expected value) are what pins the oracle."""
import math
import os

import numpy as np
import pytest

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200.scene_config import SceneGraph
from oracle import oracle as O
from tests.golden.make_golden import GOLDEN_SCENES, RENDER_H, RENDER_SEED, RENDER_SPP, RENDER_W, texture_graph
from tests.scenes_util import load

GOLDEN = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden.npz"))
MISS = 0xFFFFFFFF


def one(graph, o, d, tmin=0.001, tmax=float("inf")):
    sc = O.OracleScene(graph)
    h, _ = sc.trace_rays(np.array([list(o) + list(d)], dtype=np.float64), tmin, tmax)
    return h[0]


def simple_graph(objects, mat_kind=A.MAT_LAMBERTIAN, param=0.0, color=(0.5, 0.5, 0.5)):
    g = SceneGraph()
    t = g.add_texture(kind=A.TEX_SOLID, color=color)
    m = g.add_material(mat_kind, t, param)
    ids = [g.add_object(k, m, v=v) for k, v in objects]
    g.root = g.add_object(A.OBJ_GROUP, children=ids)
    return g


# ---------------------------------------------------------------- RNG
def test_philox4x32_10_known_answers():
    # Random123 kat_vectors for philox4x32-10
    assert list(O.philox(0, 0, 0, 0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert list(O.philox(2**64 - 1, *([2**32 - 1] * 4))) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert list(O.philox(0x299f31d0a4093822, 0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344)) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    assert (GOLDEN["philox"] == np.stack([O.philox(0, 0, 0, 0, 0), O.philox(2**64 - 1, *([2**32 - 1] * 4)),
                                          O.philox(0x299f31d0a4093822, 0x243f6a88, 0x85a308d3, 0x13198a2e,
                                                   0x03707344)])).all()


def test_noise_permutation_tables_are_permutations_and_pinned():
    for s in range(8):
        p = O.perm_table(s)
        assert sorted(p.tolist()) == list(range(256))
        assert (p == GOLDEN["perm_tables"][s]).all()
    assert not (O.perm_table(0) == O.perm_table(1)).all()


# ---------------------------------------------------------------- spheres (objects/sphere.rs:105-163)
def test_unit_sphere_from_z3_hits_at_t2_exactly():
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 1))])
    h = one(g, (0, 0, 3), (0, 0, -1))
    assert h["t"] == 2.0 and h["front_face"] == 1
    assert h["point"].tolist() == [0, 0, 1] and h["normal"].tolist() == [0, 0, 1]
    # uv: theta = acos(-0) = pi/2 -> v = .5 ; phi = atan2(-1, 0) + pi = pi/2 -> u = .25  (sphere.rs:153-159)
    assert abs(h["uv"][0] - 0.25) < 1e-15 and abs(h["uv"][1] - 0.5) < 1e-15


def test_direction_is_not_normalised_so_t_scales():
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 1))])
    assert one(g, (0, 0, 3), (0, 0, -4))["t"] == 0.5  # quirk Q8


def test_sphere_range_is_open_plane_range_is_closed():
    # sphere root exactly at tmin is rejected (surrounds, sphere.rs:133), the far root is taken instead
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 1))])
    h = one(g, (0, 0, 3), (0, 0, -1), tmin=2.0)
    assert h["t"] == 4.0 and h["front_face"] == 0
    # plane hit exactly at tmin / tmax is accepted (contains, plane.rs:150)  -- quirk Q5
    q = simple_graph([(A.OBJ_QUAD, (-1, -1, 0, 2, 0, 0, 0, 2, 0))])
    assert one(q, (0, 0, 2), (0, 0, -1), tmin=2.0)["t"] == 2.0
    assert one(q, (0, 0, 2), (0, 0, -1), tmin=0.001, tmax=2.0)["t"] == 2.0
    assert one(q, (0, 0, 2), (0, 0, -1), tmin=0.001, tmax=1.999)["object"] == MISS


def test_inside_sphere_gives_back_face_and_flipped_normal():
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 2))])
    h = one(g, (0, 0, 0), (1, 0, 0))
    assert h["t"] == 2.0 and h["front_face"] == 0 and h["normal"].tolist() == [-1, 0, 0]


# ---------------------------------------------------------------- planes (objects/plane.rs:141-174)
def test_quad_edges_inclusive_triangle_edges_exclusive():
    quad = simple_graph([(A.OBJ_QUAD, (0, 0, 0, 1, 0, 0, 0, 1, 0))])
    tri = simple_graph([(A.OBJ_TRIANGLE, (0, 0, 0, 1, 0, 0, 0, 1, 0))])
    for x, y in [(0, 0), (1, 1), (1, 0), (0, 0.5), (0.5, 1)]:  # corners and edges: alpha/beta == 0 or 1
        assert one(quad, (x, y, 1), (0, 0, -1))["t"] == 1.0
    assert one(quad, (1.0000001, 0.5, 1), (0, 0, -1))["object"] == MISS
    for x, y in [(0, 0), (0.5, 0), (0, 0.5), (0.5, 0.5)]:      # triangle: strictly inside only (:28-30)
        assert one(tri, (x, y, 1), (0, 0, -1))["object"] == MISS
    h = one(tri, (0.25, 0.25, 1), (0, 0, -1))
    assert h["t"] == 1.0 and h["uv"].tolist() == [0.25, 0.25]


def test_plane_parallel_ray_misses_by_denominator_threshold():
    quad = simple_graph([(A.OBJ_QUAD, (0, 0, 0, 1, 0, 0, 0, 1, 0))])
    assert one(quad, (0.5, 0.5, 1), (1, 0, -0.9e-8))["object"] == MISS  # |denom| < 1e-8 (plane.rs:144)
    assert one(quad, (0.5, 0.5, 1e-7), (0, 0, -1.1e-8))["object"] != MISS


def test_front_face_sign_convention():
    quad = simple_graph([(A.OBJ_QUAD, (0, 0, 0, 1, 0, 0, 0, 1, 0))])  # normal = +z
    a = one(quad, (0.5, 0.5, 1), (0, 0, -1))
    b = one(quad, (0.5, 0.5, -1), (0, 0, 1))
    assert a["front_face"] == 1 and a["normal"].tolist() == [0, 0, 1]
    assert b["front_face"] == 0 and b["normal"].tolist() == [0, 0, -1]


# ---------------------------------------------------------------- BVH (objects/object.rs:41-121, aabb.rs)
def test_equal_t_tie_goes_to_the_later_leaf():
    # two coplanar quads, identical t: the right child wins (object.rs:110-114)  -- quirk Q6
    g = simple_graph([(A.OBJ_QUAD, (0, 0, 0, 1, 0, 0, 0, 1, 0)), (A.OBJ_QUAD, (0, 0, 0, 1, 0, 0, 0, 1, 0))])
    h = one(g, (0.5, 0.5, 1), (0, 0, -1))
    assert h["object"] == 1
    g3 = simple_graph([(A.OBJ_QUAD, (0, 0, 0, 1, 0, 0, 0, 1, 0))] * 5)
    assert one(g3, (0.5, 0.5, 1), (0, 0, -1))["object"] == 4  # stable sort keeps order; last leaf wins


def test_axis_parallel_rays_through_the_slab_test():
    # d has zero components: (min-o)/0 = +-inf, and 0/0 = NaN when the origin lies on a slab plane
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 1)), (A.OBJ_SPHERE, (3, 0, 0, 1)), (A.OBJ_SPHERE, (6, 0, 0, 1))])
    assert one(g, (-5, 0, 0), (1, 0, 0))["t"] == 4.0
    assert one(g, (3, 5, 0), (0, -1, 0))["object"] == 1
    assert one(g, (3, 5, 5), (0, -1, 0))["object"] == MISS
    # origin exactly on the bbox face of the whole scene (x = -1): NaN on the x axis must not kill the hit
    h = one(g, (-1, 5, 0), (0, -1, 0))
    assert h["object"] == MISS or h["object"] == 0  # tangent graze: pinned below by the golden file, not by hand


def test_single_object_scene_has_no_box_test():
    # Leaf(Some(o)) forwards straight to the object (object.rs:95-97)  -- quirk Q7
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 1))])
    assert one(g, (0, 0, 3), (0, 0, -1))["object"] == 0


def test_empty_scene_misses():
    g = SceneGraph()
    g.root = g.add_object(A.OBJ_GROUP, children=[])
    assert one(g, (0, 0, 3), (0, 0, -1))["object"] == MISS


# ---------------------------------------------------------------- wrappers
def test_translate_rotate_scale_semantics():
    g = SceneGraph()
    t = g.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m = g.add_material(A.MAT_LAMBERTIAN, t)
    q = g.add_object(A.OBJ_QUAD, m, v=(0, 0, 0, 1, 0, 0, 0, 1, 0))
    tr = g.add_object(A.OBJ_TRANSLATE, children=[q], v=(10, 0, 0))
    g.root = g.add_object(A.OBJ_GROUP, children=[tr])
    h = one(g, (10.5, 0.5, 1), (0, 0, -1))
    assert h["t"] == 1.0 and h["point"].tolist() == [10.5, 0.5, 0.0]  # point mapped back (translate.rs:45-48)

    g = SceneGraph()
    t = g.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m = g.add_material(A.MAT_LAMBERTIAN, t)
    q = g.add_object(A.OBJ_QUAD, m, v=(-1, -1, 0, 2, 0, 0, 0, 2, 0))   # normal +z
    ry = g.add_object(A.OBJ_ROTATE_Y, children=[q], v=(math.pi / 2,))
    g.root = g.add_object(A.OBJ_GROUP, children=[ry])
    h = one(g, (3, 0, 0), (-1, 0, 0))  # +z rotated by +90deg about y faces +x
    assert abs(h["t"] - 3.0) < 1e-12 and np.allclose(h["normal"], [1, 0, 0], atol=1e-12)  # normal rotated (rotate.rs:103)

    g = SceneGraph()
    t = g.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m = g.add_material(A.MAT_LAMBERTIAN, t)
    s = g.add_object(A.OBJ_SPHERE, m, v=(0, 0, 0, 1))
    sc = g.add_object(A.OBJ_SCALE, children=[s], v=(2, 1, 1))
    g.root = g.add_object(A.OBJ_GROUP, children=[sc])
    h = one(g, (1, 5, 0), (0, -1, 0))
    # object space: o=(0.5,5,0) hits the unit sphere at y=sqrt(.75); world point x scaled back to 1;
    # the normal stays the OBJECT-space unit normal (0.5, .866, 0): Scale does not touch it (quirk Q4)
    assert np.allclose(h["point"], [1.0, math.sqrt(0.75), 0.0], atol=1e-12)
    assert np.allclose(h["normal"], [0.5, math.sqrt(0.75), 0.0], atol=1e-12)


def test_wrapper_chain_four_levels_deep():
    """Translate / Scale / Translate / Scale nested four instance levels deep (each level's group also holds a far-away
    filler, so no group forwards to its only child), around a unit sphere and a tilted quad.  Every value below is
    exact in f64: the ray goes in through o - offset (translate.rs:37-49) and the inverse scale matrix
    (scale.rs:49, 68-80: halving, quartering, doubling), the point comes back through the scale matrix and + offset.
    The normal is the OBJECT-space normal at both Scale levels (quirk Q4, scale.rs:68-80 leaves it alone): an inverse
    transpose through the non-uniform scales would tilt the quad's (0, -1, 1)/sqrt(2) to (0, -4, 1)/sqrt(17)."""
    g = SceneGraph()
    t = g.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m = g.add_material(A.MAT_LAMBERTIAN, t)
    sphere = g.add_object(A.OBJ_SPHERE, m, v=(0, 0, 0, 1))
    quad = g.add_object(A.OBJ_QUAD, m, v=(3, 0, 0, 1, 0, 0, 0, 1, 1))       # normal (0, -1, 1)/sqrt(2)
    inner = g.add_object(A.OBJ_GROUP, children=[sphere, quad])
    for kind, v in ((A.OBJ_SCALE, (1, 0.5, 1)), (A.OBJ_TRANSLATE, (0, 1, 0)), (A.OBJ_SCALE, (2, 2, 4)),
                    (A.OBJ_TRANSLATE, (4, 0, 0))):                          # innermost (level 3) first
        filler = g.add_object(A.OBJ_SPHERE, m, v=(-100, 0, 0, 1))
        inner = g.add_object(A.OBJ_GROUP, children=[g.add_object(kind, children=[inner], v=v), filler])
    g.root = inner
    # world -> object: (4, 2, 20) - (4, 0, 0) = (0, 2, 20); / (2, 2, 4) = (0, 1, 5); - (0, 1, 0) = (0, 0, 5);
    # / (1, .5, 1) = (0, 0, 5).  Direction (0, 0, -1) -> (0, 0, -.25).  Sphere (sphere.rs:114-135): a = 1/16,
    # h = 1.25, c = 24, disc = 1/16, t = (1.25 - .25) * 16 = 16.  Object point (0, 0, 1) -> (0, 0, 1) -> (0, 1, 1)
    # -> (0, 2, 4) -> (4, 2, 4) = (4, 2, 20) + 16 (0, 0, -1).
    h = one(g, (4, 2, 20), (0, 0, -1))
    assert h["object"] == sphere and h["t"] == 16.0 and h["front_face"] == 1
    assert h["point"].tolist() == [4.0, 2.0, 4.0] and h["normal"].tolist() == [0.0, 0.0, 1.0]
    # object ray (3.5, .5, 5) + t (0, 0, -.25) meets the quad's plane z = y at z = .5, t = 18, alpha = beta = .5;
    # back out: (3.5, .25, .5) -> (3.5, 1.25, .5) -> (7, 2.5, 2) -> (11, 2.5, 2) = (11, 2.5, 20) + 18 (0, 0, -1)
    h = one(g, (11, 2.5, 20), (0, 0, -1))
    s = 1.0 / math.sqrt(2.0)
    assert h["object"] == quad and abs(h["t"] - 18.0) < 1e-12 and h["front_face"] == 1
    assert np.allclose(h["point"], [11.0, 2.5, 2.0], rtol=0, atol=1e-12)
    assert np.allclose(h["normal"], [0.0, -s, s], rtol=0, atol=1e-15)
    assert np.allclose(h["uv"], [0.5, 0.5], rtol=0, atol=1e-12)


# ---------------------------------------------------------------- camera + shading quirks through tiny renders
def _render_const(graph, **cam):
    for k, v in cam.items():
        setattr(graph.camera, k, v)
    sc = O.OracleScene(graph)
    img, cnt = sc.render(O.camera_build(graph.camera.to_builder_config()), seed=1)
    return img, cnt


def test_light_seen_directly_is_dimmed_to_one():  # quirk Q3 (diffuse_light.rs:68-72)
    g = simple_graph([(A.OBJ_QUAD, (-50, -50, -1, 100, 0, 0, 0, 100, 0))], mat_kind=A.MAT_DIFFUSE_LIGHT, param=15.0,
                     color=(0.5, 0.25, 1.0))
    img, cnt = _render_const(g, width=4, height=4, samples_per_pixel=3, ray_max_bounces=5, look_from=(0, 0, 0),
                             look_at=(0, 0, -1), field_of_view=40.0, background_color=(0, 0, 0))
    assert np.allclose(img, [0.5, 0.25, 1.0], atol=1e-7)  # x1, not x15
    assert cnt["segments"] == cnt["paths"]                 # lights do not scatter


def test_background_is_constant_and_depth_zero_is_black():  # quirk Q10, camera.rs:276-278
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, -1000, 1))])
    img, _ = _render_const(g, width=3, height=2, samples_per_pixel=2, ray_max_bounces=4, look_from=(0, 0, 0),
                           look_at=(0, 0, 1), background_color=(0.7, 0.8, 1.0))
    assert np.allclose(img, [0.7, 0.8, 1.0], atol=1e-7)
    img0, cnt0 = _render_const(g, ray_max_bounces=0)
    assert (img0 == 0).all() and cnt0["segments"] == 0


def test_closed_white_sphere_leaks_because_scatter_is_not_a_unit_offset():
    # quirk Q1 (vector.rs:67): random_in_unit_sphere returns p/|p|^2 with length >= 1, so normal + v can point
    # THROUGH the surface.  Inside a closed albedo-1 sphere a textbook Lambertian would never escape (every path
    # would run max_bounces segments and return black); the reference's sampler leaks to the white background.
    g = simple_graph([(A.OBJ_SPHERE, (0, 0, 0, 5))], color=(1, 1, 1))
    img, cnt = _render_const(g, width=4, height=4, samples_per_pixel=16, ray_max_bounces=7, look_from=(0, 0, 0),
                             look_at=(0, 0, -1), background_color=(1, 1, 1))
    assert cnt["paths"] == 256 and cnt["paths"] < cnt["segments"] < 7 * cnt["paths"]
    # each path contributes exactly 0 (depth cap) or 1 (escaped with throughput 1): pixel values are k/16
    assert np.allclose(img * 16, np.round(img * 16), atol=1e-5) and 0.3 < img.mean() < 1.0


def _two_material_scene(first_kind, first_param, first_color, light_quad, light_color=(1.0, 1.0, 1.0), intensity=4.0):
    """A big quad in the plane y = 0 with the material under test, and one small light quad."""
    g = SceneGraph()
    t0 = g.add_texture(kind=A.TEX_SOLID, color=first_color)
    m0 = g.add_material(first_kind, t0, first_param)
    t1 = g.add_texture(kind=A.TEX_SOLID, color=light_color)
    m1 = g.add_material(A.MAT_DIFFUSE_LIGHT, t1, intensity)
    floor = g.add_object(A.OBJ_QUAD, m0, v=(-5, 0, -5, 0, 0, 10, 10, 0, 0))   # u x v = +y: the front face looks up
    light = g.add_object(A.OBJ_QUAD, m1, v=light_quad)
    g.root = g.add_object(A.OBJ_GROUP, children=[floor, light])
    return g


def test_metal_without_fuzz_is_a_perfect_mirror():
    """metal.rs:73-91: scattered = reflect(dir, n).normalize() + fuzz * random_in_unit_sphere; colour = texture.
    A ray coming down at 45 degrees onto the plane y = 0 leaves along (1, 1, 0) and meets a light placed exactly
    there; seen through a bounce the light counts with its intensity (diffuse_light.rs:63-75)."""
    light_at = lambda cx, cy: (cx - 0.35, cy + 0.35, -0.5, 0.7, -0.7, 0.0, 0.0, 0.0, 1.0)   # noqa: E731 — faces the origin
    cam = dict(width=1, height=1, samples_per_pixel=1, ray_max_bounces=5, look_from=(-2.0, 2.0, 0.0),
               look_at=(0.0, 0.0, 0.0), field_of_view=1.0, background_color=(0.0, 0.0, 0.0))
    g = _two_material_scene(A.MAT_METAL, 0.0, (0.8, 0.6, 0.2), light_at(2.0, 2.0))
    img, cnt = _render_const(g, **cam)
    assert np.allclose(img[0, 0], [0.8 * 4.0, 0.6 * 4.0, 0.2 * 4.0], rtol=1e-6) and cnt["segments"] == 2
    # the same light one unit off the mirror direction is not seen: the path ends on the (black) background
    g = _two_material_scene(A.MAT_METAL, 0.0, (0.8, 0.6, 0.2), light_at(3.2, 0.8))
    img, cnt = _render_const(g, **cam)
    assert (img == 0).all() and cnt["segments"] == 2
    # with fuzz the direction is perturbed by fuzz * p/|p|^2 (|p/|p|^2| >= 1): at fuzz 0.2 the 0.7-wide light two
    # units away is still hit by some samples but no longer by all
    g = _two_material_scene(A.MAT_METAL, 0.2, (1.0, 1.0, 1.0), light_at(2.0, 2.0))
    img, cnt = _render_const(g, **dict(cam, samples_per_pixel=400, field_of_view=0.01))
    assert 0.05 * 4.0 < img[0, 0, 0] < 0.95 * 4.0


def test_dielectric_follows_snell_and_schlick():
    """dielectric.rs:39-67.  45 degrees onto glass (index 1.5) from outside: ri = 1/1.5, sin(t) = sin(45)/1.5, the
    refracted ray leaves the origin along (sin t, -cos t, 0); reflectance (Schlick, :13-19) r0 = ((1-ri)/(1+ri))^2
    = 0.04, R = r0 + (1-r0)(1-cos 45)^5 = 0.04207; the ray reflects iff R > u for one uniform draw."""
    sin_t = math.sin(math.radians(45.0)) / 1.5
    cos_t = math.sqrt(1.0 - sin_t * sin_t)
    x_hit = 2.0 * sin_t / cos_t                                   # where the refracted ray crosses y = -2
    light_below = lambda cx: (cx - 0.2, -2.0, -0.2, 0.4, 0.0, 0.0, 0.0, 0.0, 0.4)   # noqa: E731
    R = 0.04 + 0.96 * (1.0 - math.cos(math.radians(45.0))) ** 5
    cam = dict(width=1, height=1, samples_per_pixel=4000, ray_max_bounces=5, look_from=(-2.0, 2.0, 0.0),
               look_at=(0.0, 0.0, 0.0), field_of_view=0.01, background_color=(0.0, 0.0, 0.0))
    g = _two_material_scene(A.MAT_DIELECTRIC, 1.5, (1.0, 1.0, 1.0), light_below(x_hit), intensity=1.0)
    img, cnt = _render_const(g, **cam)
    refracted = float(img[0, 0, 0])          # attenuation 1 (:61), light 1: the pixel is the refracted fraction
    assert abs(refracted - (1.0 - R)) < 4.0 * math.sqrt(R * (1.0 - R) / 4000.0) + 1e-3
    assert cnt["segments"] == 2 * cnt["paths"]
    # a light where a straight (unrefracted) continuation would land, x = 2 at y = -2, stays dark
    g = _two_material_scene(A.MAT_DIELECTRIC, 1.5, (1.0, 1.0, 1.0), light_below(2.0), intensity=1.0)
    img, _ = _render_const(g, **cam)
    assert float(img[0, 0, 0]) == 0.0
    # from inside the glass beyond the critical angle (asin(1/1.5) = 41.8 deg) everything reflects: the ray comes
    # up at 45 degrees against the underside and is mirrored back down onto a light below
    cam_in = dict(cam, look_from=(-2.0, -2.0, 0.0), samples_per_pixel=200)
    g = _two_material_scene(A.MAT_DIELECTRIC, 1.5, (1.0, 1.0, 1.0), light_below(2.0), intensity=1.0)
    img, _ = _render_const(g, **cam_in)
    assert abs(float(img[0, 0, 0]) - 1.0) < 1e-6


def _lambertian_leak_scene():
    """A Lambertian floor (front face up) over a huge light: only scattered rays that go THROUGH the floor see it."""
    g = _two_material_scene(A.MAT_LAMBERTIAN, 0.0, (0.5, 0.5, 0.5), (-500.0, -1.0, -500.0, 1000.0, 0, 0, 0, 0, 1000.0),
                            intensity=2.0)
    return g


def test_lambertian_scatter_is_normal_plus_p_over_p_squared():
    """lambertian.rs:39-55 + vector.rs:61-70 (quirk Q1): the scatter direction is n + p/|p|^2 with p uniform in the
    unit ball, so |offset| = 1/|p| >= 1 and the ray dives below the surface iff cos(theta) < -|p|:
    P = int_0^1 3r^2 (1-r)/2 dr = 1/8.  (The textbook n + unit vector never goes below.)  With a light under the floor
    and a black sky the pixel is albedo * emission * 1/8."""
    g = _lambertian_leak_scene()
    n = 20000
    img, cnt = _render_const(g, width=1, height=1, samples_per_pixel=n, ray_max_bounces=2, look_from=(-2.0, 2.0, 0.0),
                             look_at=(0.0, 0.0, 0.0), field_of_view=0.01, background_color=(0.0, 0.0, 0.0))
    p = float(img[0, 0, 0]) / (0.5 * 2.0)
    assert abs(p - 0.125) < 4.0 * math.sqrt(0.125 * 0.875 / n)
    assert cnt["segments"] == 2 * cnt["paths"]


# ---------------------------------------------------------------- golden fixtures (pin the oracle)
@pytest.mark.parametrize("name", GOLDEN_SCENES + ["_textures"])
def test_oracle_reproduces_golden(name):
    key = name.split(".")[0].replace("-", "_")
    if name == "_textures":
        g = texture_graph()
        g.camera.width, g.camera.height, g.camera.samples_per_pixel = RENDER_W, RENDER_H, RENDER_SPP
    else:
        g = load(name, width=RENDER_W, height=RENDER_H, samples_per_pixel=RENDER_SPP)
    sc = O.OracleScene(g)
    hits, _ = sc.trace_rays(GOLDEN[f"{key}__rays"])
    gold = GOLDEN[f"{key}__hits"]
    assert (hits["object"] == gold["object"]).all()
    assert (hits["t"] == gold["t"]).all()
    assert np.array_equal(hits["point"], gold["point"]) and np.array_equal(hits["normal"], gold["normal"])
    cam = O.camera_build(g.camera.to_builder_config())
    assert bytes(cam) == GOLDEN[f"{key}__camera"].tobytes()
    img, cnt = sc.render(cam, seed=RENDER_SEED)
    assert cnt["segments"] == int(GOLDEN[f"{key}__segments"][0])
    assert np.array_equal(img, GOLDEN[f"{key}__image"])


def test_oracle_textures_match_golden_and_definitions():
    g = texture_graph()
    sc = O.OracleScene(g)
    uvp = GOLDEN["tex__uvp"]
    for ti in range(len(g.textures)):
        assert np.array_equal(sc.texture_eval(ti, uvp), GOLDEN[f"tex__{ti}"])
    # checker (checker.rs:77-89): parity of trunc(u*s) + trunc(v*s), negatives saturate to 0
    chk = sc.texture_eval(2, np.array([[0.05, 0.05, 0, 0, 0], [0.15, 0.05, 0, 0, 0], [-0.5, 0.15, 0, 0, 0]]))
    assert chk[0].tolist() == [0.9, 0.1, 0.2] and chk[1].tolist() == [0.1, 0.8, 0.3] and chk[2].tolist() == [0.1, 0.8, 0.3]
    # image (image.rs:30-40): nearest texel, v flipped, value = u8/255 in f32
    img = g.images[0]
    px = sc.texture_eval(6, np.array([[0.0, 1.0, 0, 0, 0], [0.5, 0.5, 0, 0, 0], [1.0, 0.0, 0, 0, 0]]))
    assert np.array_equal(px[0], (img[0, 0].astype(np.float32) / np.float32(255)).astype(np.float64))
    assert np.array_equal(px[1], (img[4, 8].astype(np.float32) / np.float32(255)).astype(np.float64))
    assert np.array_equal(px[2], (img[7, 15].astype(np.float32) / np.float32(255)).astype(np.float64))  # clamped edge
    # noise is |fbm| in [0, 1]; marble in [0, 1]
    assert (GOLDEN["tex__3"] >= 0).all() and (GOLDEN["tex__3"] <= 1).all() and GOLDEN["tex__3"].std() > 0.01
    assert (GOLDEN["tex__4"] >= 0).all() and (GOLDEN["tex__4"] <= 1).all()


def test_oracle_render_is_deterministic_and_sample_ranges_compose():
    g = load("cornell-box-scene.json", width=24, height=16, samples_per_pixel=8)
    sc = O.OracleScene(g)
    cam = O.camera_build(g.camera.to_builder_config())
    a, ca = sc.render(cam, seed=3)
    b, _ = sc.render(cam, seed=3, n_threads=1)
    assert np.array_equal(a, b)
    lo, c1 = sc.render(cam, seed=3, sample_range=(0, 4))
    hi, c2 = sc.render(cam, seed=3, sample_range=(4, 8))
    assert c1["segments"] + c2["segments"] == ca["segments"]
    assert np.allclose((lo.astype(np.float64) + hi) / 2, a, rtol=1e-6, atol=1e-7)
    other, _ = sc.render(cam, seed=4)
    assert not np.array_equal(a, other)


def test_moving_sphere_center_follows_ray_time():
    """sphere.rs:110-111: center(t) = center + time*speed; :75-78: bbox = union of the boxes at time 0 and 1."""
    from nr_ray_tracer_b200.scene_config import SceneGraph
    g = SceneGraph()
    t = g.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m = g.add_material(A.MAT_LAMBERTIAN, t)
    s = g.add_object(A.OBJ_SPHERE, m, v=(0, 0, 0, 1, 2, 0, 0))   # speed (2, 0, 0)
    g.root = g.add_object(A.OBJ_GROUP, children=[s])
    sc = O.OracleScene(g)
    rays = np.array([[1.5, 0, 5, 0, 0, -1],     # x = 1.5: outside at time 0, inside at time 0.5 (center x = 1)
                     [0.0, 0, 5, 0, 0, -1]])    # x = 0: centre hit at time 0, miss at time 0.75 (center x = 1.5)
    h0, _ = sc.trace_rays(rays, time=0.0)
    assert np.isinf(h0["t"][0]) and h0["t"][1] == 4.0
    h5, _ = sc.trace_rays(rays, time=0.5)
    assert h5["t"][0] == 5.0 - np.sqrt(1.0 - 0.25)
    np.testing.assert_allclose(h5["normal"][0], [0.5, 0, np.sqrt(0.75)], atol=1e-15)   # (point - center(t)) normalised
    h75, _ = sc.trace_rays(rays, time=0.75)
    assert np.isinf(h75["t"][1]) and np.isfinite(h75["t"][0])
    # the render draws time per camera ray: the image of a moving sphere is a blur, not the static image
    from nr_ray_tracer_b200.scene_config import CameraConfig
    cfg = CameraConfig(width=48, height=27, samples_per_pixel=16, ray_max_bounces=4, look_from=(0.0, 0.0, 8.0),
                       look_at=(0.0, 0.0, 0.0), background_color=(0.5, 0.7, 1.0)).to_builder_config()
    cam = O.camera_build(cfg)
    moving, _ = sc.render(cam, seed=3)
    g2 = SceneGraph()
    t2 = g2.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m2 = g2.add_material(A.MAT_LAMBERTIAN, t2)
    g2.root = g2.add_object(A.OBJ_GROUP, children=[g2.add_object(A.OBJ_SPHERE, m2, v=(0, 0, 0, 1))])
    static, _ = O.OracleScene(g2).render(cam, seed=3)
    assert not np.array_equal(moving, static)
    # Some(ZERO) speed behaves exactly like None
    g3 = SceneGraph()
    t3 = g3.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m3 = g3.add_material(A.MAT_LAMBERTIAN, t3)
    g3.root = g3.add_object(A.OBJ_GROUP, children=[g3.add_object(A.OBJ_SPHERE, m3, v=(0, 0, 0, 1, 0, 0, 0))])
    same, _ = O.OracleScene(g3).render(cam, seed=3)
    assert np.array_equal(same, static)


# ------------------------------------------------------------------ third-party arithmetic: hand-derived pins
def _noise_scene(**kw):
    g = SceneGraph()
    g.add_texture(kind=A.TEX_NOISE, **kw)
    m = g.add_material(A.MAT_LAMBERTIAN, 0)
    g.root = g.add_object(A.OBJ_GROUP, children=[g.add_object(A.OBJ_SPHERE, m, v=(0, 0, 0, 1))])
    return O.OracleScene(g)


def _at(points):
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    return np.concatenate([np.zeros((len(p), 2)), p], axis=1)


def test_perlin_is_zero_on_the_integer_lattice():
    """Gradient noise (noise 0.9.0 Perlin::get, used by textures/noise.rs:87-93): at a lattice point every corner
    offset that carries weight is the zero vector, so the value is exactly 0 — for every seed, whatever the
    permutation table holds.  With frequency 1 and an integer lacunarity all octaves sample lattice points."""
    pts = [(x, y, z) for x in (-3, 0, 1, 7) for y in (-1, 0, 2) for z in (0, 5, -4)]
    for seed in (0, 1, 12345):
        for octaves in (1, 4):
            sc = _noise_scene(seed=seed, octaves=octaves, f0=1.0, f1=2.0, f2=0.5)
            assert np.array_equal(sc.texture_eval(0, _at(pts)), np.zeros((len(pts), 3)))


def test_fbm_scale_factor_for_1_7_and_8_octaves():
    """Fbm (noise 0.9.0): result = sum_i perlin_i(p * f * lac^i) * pers^(i+1), times scale_factor = 1 / sum_{i=1..n} pers^i.
    At a point whose coordinates are all odd multiples of 1/2, with lacunarity 2, every octave but the first samples
    the integer lattice (= 0), so |fbm_n| = |perlin_0| * pers * scale_n with scale_1 = 2, scale_7 = 128/127,
    scale_8 = 256/255 for pers = 1/2 — the first octave's table (seed + 0) is the same for every n."""
    p = _at([(0.5, 1.5, 2.5), (-1.5, 0.5, 3.5), (2.5, -0.5, 0.5)])
    v = {n: _noise_scene(seed=5, octaves=n, f0=1.0, f1=2.0, f2=0.5).texture_eval(0, p)[:, 0] for n in (1, 7, 8)}
    assert (v[1] > 1e-3).any()                       # the probe points are not all zeros of octave 0
    assert np.allclose(v[7], v[1] * (64.0 / 127.0), rtol=4e-16, atol=0)
    assert np.allclose(v[8], v[1] * (128.0 / 255.0), rtol=4e-16, atol=0)
    # one octave: persistence cancels against its own scale factor (x * p * (1/p))
    w = _noise_scene(seed=5, octaves=1, f0=1.0, f1=2.0, f2=0.9).texture_eval(0, p)[:, 0]
    assert np.allclose(w, v[1], rtol=4e-16, atol=0)
    # Marble is 7 octaves at lacunarity 2*pi/3 (marble.rs:50-54): bounded by construction
    g = SceneGraph()
    g.add_texture(kind=A.TEX_MARBLE, seed=0, octaves=7, f0=0.2)
    m = g.add_material(A.MAT_LAMBERTIAN, 0)
    g.root = g.add_object(A.OBJ_GROUP, children=[g.add_object(A.OBJ_SPHERE, m, v=(0, 0, 0, 1))])
    mv = O.OracleScene(g).texture_eval(0, _at(np.random.default_rng(0).uniform(-50, 50, (500, 3))))
    assert (mv >= 0).all() and (mv <= 1).all() and mv.std() > 0.05


def test_scale_matrix_inverse_for_the_cornell_scales():
    """Scale::new (scale.rs:48-49): DMat4::from_scale(s).inverse().  For the Cornell box's two scales the cofactors and
    the determinant are exact binary fractions, so every formulation (cofactor / det, cofactor * (1 / det)) must give
    diag(4, 4, 4) and diag(4, fl(4/3), 4) with a zero translation column — checked on the product's host build
    (csrc/host_math.hpp Mat4::inverse through nrrt_xform.to_obj) and, through hits, on the oracle."""
    from nr_ray_tracer_b200 import api
    g = load("cornell-box-scene.json")
    hs = api.HostScene(g)
    scales = [hs.desc.xforms[i] for i in range(hs.desc.n_xforms) if hs.desc.xforms[i].kind == 2]
    assert len(scales) == 2
    got = sorted(tuple(x.to_obj) for x in scales)
    want = sorted([(4.0, 0, 0, 0, 4.0, 0, 0, 0, 4.0, 0, 0, 0), (4.0, 0, 0, 0, 4.0 / 3.0, 0, 0, 0, 4.0, 0, 0, 0)])
    assert got == want
    for x in scales:
        fwd = tuple(x.to_world)
        assert fwd[0] == 0.25 and fwd[8] == 0.25 and fwd[4] in (0.25, 0.75) and fwd[9:] == (0.0, 0.0, 0.0)
    # the oracle's Scale: a unit quad at z = 0 scaled by (0.25, 0.75, 0.25) is hit at u = x / 0.25, v = y / 0.75
    sg = SceneGraph()
    t = sg.add_texture(kind=A.TEX_SOLID, color=(1, 1, 1))
    m = sg.add_material(A.MAT_LAMBERTIAN, t)
    q = sg.add_object(A.OBJ_QUAD, m, v=(0, 0, 0, 1, 0, 0, 0, 1, 0))
    s = sg.add_object(A.OBJ_SCALE, children=[q], v=(0.25, 0.75, 0.25))
    sg.root = sg.add_object(A.OBJ_GROUP, children=[s])
    hit, _ = O.OracleScene(sg).trace_rays(np.array([[0.125, 0.5, 2.0, 0, 0, -1.0]]))
    assert hit["object"][0] == q and hit["t"][0] == 2.0
    assert hit["uv"][0].tolist() == [0.125 * 4.0, 0.5 * (4.0 / 3.0)]


# ------------------------------------------------------------------ the real crate's answers, when someone has dumped them
RUST_DUMP = os.path.join(os.path.dirname(__file__), "golden", "rust_dump")
RUST_NOISE_CFGS = [dict(seed=0, octaves=1, f0=1.0, f1=2.0 * math.pi / 3.0, f2=0.5),      # noise.rs defaults
                   dict(seed=0, octaves=8, f0=0.2, f1=2.0 * math.pi / 3.0, f2=0.5),      # scenes/noise.toml
                   dict(seed=3, octaves=5, f0=1.7, f1=2.1, f2=0.45), dict(seed=7, octaves=1, f0=3.0, f1=2.0 * math.pi / 3.0, f2=0.9)]
RUST_MARBLE_CFGS = [dict(seed=0, f0=1.0), dict(seed=1, f0=0.8), dict(seed=0, f0=0.2)]


def rust_dump_points():
    """Sample points of the texture dump (rust/golden-dump reads them from texture_points.bin)."""
    rng = np.random.default_rng(2718)
    return np.concatenate([rng.uniform(-40, 40, (400, 3)), rng.uniform(-1, 1, (100, 3)),
                           np.array([[0.0, 0.0, 0.0], [1.0, 2.0, 3.0], [0.5, 1.5, 2.5], [-7.25, 3.125, 11.0]])])


@pytest.mark.skipif(not os.path.isdir(RUST_DUMP) or not os.path.exists(os.path.join(RUST_DUMP, "perm.bin")),
                    reason="tests/golden/rust_dump/ absent: run rust/golden-dump on a machine with cargo (rust/README.md); "
                           "until then the oracle's parity with the Rust crate is unpinned")
def test_against_rust_dump():
    """The oracle against known answers dumped from the REAL nr-ray-tracer crates (rust/golden-dump): BVH::hit on the
    golden rays of every scene the current reference loader accepts, noise 0.9.0 permutation tables, Texture::get_color
    of the noise / marble textures, DMat4::inverse.  Bit-exact, except transcendental-dependent values (2 ulp)."""
    perm = np.fromfile(os.path.join(RUST_DUMP, "perm.bin"), dtype=np.uint8).reshape(-1, 256)
    for seed in range(perm.shape[0]):
        assert np.array_equal(perm[seed], O.perm_table(seed)), f"permutation table, seed {seed}"
    pts = _at(rust_dump_points())
    tex = np.fromfile(os.path.join(RUST_DUMP, "textures.bin"), dtype="<f8").reshape(-1, len(pts))
    rows = [_noise_scene(**c).texture_eval(0, pts)[:, 0] for c in RUST_NOISE_CFGS]
    for c in RUST_MARBLE_CFGS:
        g = SceneGraph()
        g.add_texture(kind=A.TEX_MARBLE, octaves=7, **c)
        m = g.add_material(A.MAT_LAMBERTIAN, 0)
        g.root = g.add_object(A.OBJ_GROUP, children=[g.add_object(A.OBJ_SPHERE, m, v=(0, 0, 0, 1))])
        rows.append(O.OracleScene(g).texture_eval(0, pts)[:, 0])
    assert tex.shape[0] == len(rows)
    for k, row in enumerate(rows):
        tol = 0 if k < len(RUST_NOISE_CFGS) else 4e-16      # marble goes through sin()
        assert np.allclose(tex[k], row, rtol=tol, atol=tol), f"texture config {k}"
    inv = np.fromfile(os.path.join(RUST_DUMP, "dmat4_inverse.bin"), dtype="<f8").reshape(-1, 16)
    assert inv[0].tolist() == [4.0, 0, 0, 0, 0, 4.0, 0, 0, 0, 0, 4.0, 0, 0, 0, 0, 1.0]
    assert inv[1].tolist() == [4.0, 0, 0, 0, 0, 4.0 / 3.0, 0, 0, 0, 0, 4.0, 0, 0, 0, 0, 1.0]
    checked = 0
    for name in GOLDEN_SCENES:
        f = os.path.join(RUST_DUMP, f"{name}.hits.bin")
        if not os.path.exists(f):
            continue                                            # legacy-schema scene / the teapot stand-in
        rust = np.fromfile(f, dtype="<f8").reshape(-1, 11)
        key = name.split(".")[0].replace("-", "_")
        ref = GOLDEN[f"{key}__hits"]
        hit_r = ref["object"] != 0xFFFFFFFF
        assert np.array_equal(rust[:, 0] == 1.0, hit_r), name
        assert np.array_equal(rust[hit_r, 1], ref["t"][hit_r]), name
        assert np.array_equal(rust[hit_r, 10] == 1.0, ref["front_face"][hit_r] == 1), name
        assert np.allclose(rust[hit_r, 2:5], ref["point"][hit_r], rtol=0, atol=0), name
        assert np.allclose(rust[hit_r, 5:8], ref["normal"][hit_r], rtol=0, atol=0), name
        assert np.allclose(rust[hit_r, 8:10], ref["uv"][hit_r], rtol=4e-16, atol=4e-16), name   # acos / atan2
        checked += 1
    assert checked >= 2


def test_render_chunked_is_render_with_the_sum_reassociated():
    """oracle_render_chunked: one chunk, or one sample per chunk, is the plain sequential sum of render(); any other
    split changes at most the last bits (same paths, same counts)."""
    g = load("spheres.toml", width=40, height=22, samples_per_pixel=24)
    sc = O.OracleScene(g)
    cam = O.camera_build(g.camera.to_builder_config())
    a, ca = sc.render(cam, seed=3)
    b, cb = sc.render_chunked(cam, [0, 24], seed=3)
    c, cc = sc.render_chunked(cam, list(range(25)), seed=3)
    d, cd = sc.render_chunked(cam, [0, 5, 10, 15, 20, 24], seed=3)
    assert np.array_equal(a, b) and np.array_equal(a, c) and ca == cb == cc == cd
    assert np.allclose(a, d, rtol=3e-7, atol=0)
    with pytest.raises(ValueError):
        sc.render_chunked(cam, [0, 5, 5, 24], seed=3)
