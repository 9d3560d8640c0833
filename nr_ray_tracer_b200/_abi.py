"""ctypes mirror of include/nrrt.h (the C ABI).  Data definitions only.

Field order and types must match the header exactly; tests/test_abi.py checks the
struct sizes against the values the compiled library reports.
"""
import ctypes as C

ABI_VERSION = 4
BUILD_REFERENCE, BUILD_SAH = 0, 1

# status codes
OK, ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_NO_SCENE, ERR_LIMIT, ERR_IO = 0, -1, -2, -3, -4, -5, -6

# object kinds
OBJ_SPHERE, OBJ_QUAD, OBJ_TRIANGLE, OBJ_GROUP, OBJ_TRANSLATE, OBJ_ROTATE_X, OBJ_ROTATE_Y, OBJ_ROTATE_Z, OBJ_SCALE = range(9)
# material kinds
MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_DIFFUSE_LIGHT = range(4)
# texture kinds
TEX_SOLID, TEX_CHECKER, TEX_IMAGE, TEX_NOISE, TEX_MARBLE = range(5)

REF_NODE, REF_SPHERE, REF_PLANE, REF_INSTANCE, REF_EMPTY = 0, 1, 2, 3, 7
REF_NONE = 0xFFFFFFFF
REF_TYPE_SHIFT = 29
REF_INDEX_MASK = 0x1FFFFFFF

TRACE_ORDERED, TRACE_VISIT_ALL, TRACE_DEVICE_BUFFERS, TRACE_COUNT, TRACE_COMPACT = 0, 1, 2, 4, 8
MODE_WAVEFRONT, MODE_MEGAKERNEL, MODE_FUSED, MODE_POOL, MODE_AUTO = 0, 1, 2, 3, 4
MODE_NAMES = {0: "wavefront", 1: "megakernel", 2: "fused", 3: "pool", 4: "auto"}
RENDER_OUT_HOST, RENDER_OUT_DEVICE, RENDER_COUNT, RENDER_OUT_PACKED = 0, 1, 2, 4
MAX_INSTANCE_DEPTH = 4

u32, u64, f64, f32 = C.c_uint32, C.c_uint64, C.c_double, C.c_float


class Object(C.Structure):
    _fields_ = [("kind", u32), ("material", u32), ("first_child", u32), ("n_children", u32), ("v", f64 * 9)]


class Material(C.Structure):
    _fields_ = [("kind", u32), ("texture", u32), ("param", f64)]


class Texture(C.Structure):
    _fields_ = [("kind", u32), ("a", u32), ("b", u32), ("seed", u32), ("octaves", u32), ("_pad", u32),
                ("color", f64 * 3), ("f0", f64), ("f1", f64), ("f2", f64)]


class Image(C.Structure):
    _fields_ = [("width", u32), ("height", u32), ("rgb", C.c_void_p)]


class GraphDesc(C.Structure):
    _fields_ = [("n_objects", u32), ("objects", C.POINTER(Object)),
                ("n_child_ids", u32), ("child_ids", C.POINTER(u32)),
                ("n_materials", u32), ("materials", C.POINTER(Material)),
                ("n_textures", u32), ("textures", C.POINTER(Texture)),
                ("n_images", u32), ("images", C.POINTER(Image)),
                ("root", u32)]


class CameraConfig(C.Structure):
    _fields_ = [("width", u32), ("height", u32), ("samples_per_pixel", u32), ("ray_max_bounces", u32),
                ("background", f64 * 3), ("look_from", f64 * 3), ("look_at", f64 * 3), ("view_up", f64 * 3),
                ("defocus_angle", f64), ("focus_dist", f64), ("field_of_view", f64)]


class Camera(C.Structure):
    _fields_ = [("width", u32), ("height", u32), ("samples_per_pixel", u32), ("ray_max_bounces", u32),
                ("background", f64 * 3), ("look_from", f64 * 3),
                ("defocus_disk_u", f64 * 3), ("defocus_disk_v", f64 * 3),
                ("pixel_delta_u", f64 * 3), ("pixel_delta_v", f64 * 3), ("viewport_top_left", f64 * 3)]


class Node(C.Structure):
    _fields_ = [("lo", (f32 * 3) * 2), ("hi", (f32 * 3) * 2), ("child", u32 * 2), ("_pad", u32 * 2)]


class Box(C.Structure):
    _fields_ = [("lo", f64 * 3), ("hi", f64 * 3)]


class WNode(C.Structure):
    _fields_ = [("lo", (f32 * 4) * 3), ("hi", (f32 * 4) * 3), ("child", u32 * 4), ("meta", u32 * 4)]


WNODE_GATED = 1


class Xform(C.Structure):
    _fields_ = [("kind", u32), ("_pad", u32), ("to_obj", f64 * 12), ("to_world", f64 * 12)]


class Instance(C.Structure):
    _fields_ = [("first_xform", u32), ("n_xforms", u32), ("inner", u32), ("_pad", u32), ("inner_box", Box)]


class SceneDesc(C.Structure):
    _fields_ = [
        ("abi_version", u32),
        ("n_nodes", u32), ("nodes", C.POINTER(Node)), ("child_boxes", C.POINTER(Box)),
        ("root", u32), ("root_box", Box),
        ("n_spheres", u32), ("sphere_rec", C.POINTER(f64)),
        ("sphere_material", C.POINTER(u32)), ("sphere_order", C.POINTER(u32)), ("sphere_object", C.POINTER(u32)),
        ("n_planes", u32), ("plane_rec", C.POINTER(f64)),
        ("plane_material", C.POINTER(u32)), ("plane_order", C.POINTER(u32)), ("plane_object", C.POINTER(u32)),
        ("n_instances", u32), ("instances", C.POINTER(Instance)), ("instance_order", C.POINTER(u32)),
        ("n_xforms", u32), ("xforms", C.POINTER(Xform)),
        ("n_materials", u32), ("materials", C.POINTER(Material)),
        ("n_textures", u32), ("textures", C.POINTER(Texture)),
        ("n_images", u32), ("images", C.POINTER(Image)),
        ("max_stack", u32),
        ("sphere_speed", C.POINTER(f64)),
        ("n_wnodes", u32), ("wnodes", C.POINTER(WNode)), ("wide_boxes", C.POINTER(Box)),
        ("wide_root", u32), ("instance_wide_inner", C.POINTER(u32)),
    ]


class Hit(C.Structure):
    _fields_ = [("t", f64), ("point", f64 * 3), ("normal", f64 * 3), ("uv", f64 * 2),
                ("prim", u32), ("material", u32), ("front_face", u32), ("object", u32), ("depth", u32),
                ("inst", u32 * MAX_INSTANCE_DEPTH), ("_pad", u32)]


class HitCompact(C.Structure):
    _fields_ = [("t", f64), ("prim", u32), ("depth_inst0", u32)]


class TraceStats(C.Structure):
    _fields_ = [("node_visits", u64), ("box_exact", u64), ("prim_tests", u64), ("kernel_ms", f64)]


class RenderOpts(C.Structure):
    _fields_ = [("seed", u64), ("mode", u32), ("rank", u32), ("world", u32), ("rows_per_block", u32),
                ("max_slots", u32), ("flags", u32)]


class RenderStats(C.Structure):
    _fields_ = [("paths", u64), ("segments", u64), ("launches", u64), ("device_ms", f64), ("extend_ms", f64),
                ("extend_launches", u64), ("pixels", u32), ("mode", u32),
                ("node_visits", u64), ("box_exact", u64), ("prim_tests", u64), ("inst_entries", u64),
                ("inst_misses", u64)]


class AdaptiveOpts(C.Structure):
    _fields_ = [("rel_error", f64), ("abs_error", f64), ("min_samples", u32), ("_pad", u32)]


class CameraFile(C.Structure):
    _fields_ = [("present", u32), ("width", u32), ("height", u32), ("samples_per_pixel", u32), ("ray_max_bounces", u32),
                ("_pad", u32), ("aspect_ratio", f64), ("background", f64 * 3), ("look_at", f64 * 3),
                ("look_from", f64 * 3), ("view_up", f64 * 3), ("field_of_view_deg", f64), ("defocus_angle_deg", f64),
                ("focus_distance", f64)]


CAM_WIDTH, CAM_HEIGHT, CAM_ASPECT_RATIO, CAM_BACKGROUND, CAM_LOOK_AT, CAM_LOOK_FROM, CAM_VIEW_UP, CAM_FOV, \
    CAM_DEFOCUS, CAM_FOCUS, CAM_SPP, CAM_BOUNCES = (1 << i for i in range(12))

PROGRESS_FN = C.CFUNCTYPE(None, u64, u64, C.c_void_p)

# numpy dtype of nrrt_hit for zero-copy result arrays
import numpy as _np  # noqa: E402

HIT_DTYPE = _np.dtype([("t", "<f8"), ("point", "<f8", (3,)), ("normal", "<f8", (3,)), ("uv", "<f8", (2,)),
                       ("prim", "<u4"), ("material", "<u4"), ("front_face", "<u4"), ("object", "<u4"),
                       ("depth", "<u4"), ("inst", "<u4", (MAX_INSTANCE_DEPTH,)), ("_pad", "<u4")])
assert HIT_DTYPE.itemsize == C.sizeof(Hit)
