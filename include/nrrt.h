/*
 * nrrt.h — C ABI of the B200-native path-tracing hot path of nr-ray-tracer.
 *
 * The reference has no FFI boundary: its hot path is the generic Rust call
 *   Scene::render(&self, progress) -> Rgb32FImage        (packages/ray-tracer-lib/src/scene.rs:13-18)
 *     -> Camera::render(&self, hitable, progress)        (packages/ray-tracer-lib/src/camera.rs:302-343)
 * whose only caller is  packages/ray-tracer/src/commands/render.rs:59.
 * This header defines the boundary a Rust `-sys` crate would bind (see
 * INTEGRATION.md): plain pointers and sizes only, caller-owned host buffers,
 * every device allocation owned by the context, integer status codes.
 *
 * Two layers:
 *   1. "graph" layer  (nrrt_graph_*)  — a description of the reference's object
 *      graph (what CLI scene_config.rs:278-380 builds): spheres, quads,
 *      triangles, groups (= BVH::from), translate/rotate/scale wrappers,
 *      materials, textures.  nrrt_host_build() runs the reference's BVH build
 *      (objects/object.rs:41-73) on the host and flattens the tree into ...
 *   2. "flat" layer   (nrrt_scene_desc) — the structure-of-arrays device layout
 *      (64-byte two-child f32 nodes + exact f64 boxes, aligned primitive records, instance
 *      transform chains, material/texture tables) that nrrt_scene_upload()
 *      copies to HBM and the CUDA kernels traverse.
 *
 * All geometry is f64 like the reference; f32 appears only in conservative
 * culling boxes and the output framebuffer.
 */
#ifndef NRRT_H
#define NRRT_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRRT_ABI_VERSION 4

/* ---- status codes ------------------------------------------------------ */
enum {
    NRRT_OK = 0,
    NRRT_ERR_INVALID = -1,   /* bad argument / malformed scene            */
    NRRT_ERR_CUDA = -2,      /* CUDA runtime failure (see nrrt_last_error) */
    NRRT_ERR_NO_DEVICE = -3, /* no usable GPU: there is NO CPU fallback    */
    NRRT_ERR_NO_SCENE = -4,  /* render/trace before nrrt_scene_upload      */
    NRRT_ERR_LIMIT = -5,     /* scene exceeds a compiled-in limit          */
    NRRT_ERR_IO = -6         /* scene file / texture could not be read     */
};

/* ======================================================================== */
/* 1. graph layer: mirror of ObjectConfig / MaterialConfig / TextureConfig  */
/*    after id resolution (CLI scene_config.rs:27-259).                     */
/* ======================================================================== */

enum nrrt_obj_kind {
    NRRT_OBJ_SPHERE = 0,    /* v[0..2]=center v[3]=radius v[4..6]=speed (SphereBuilder::with_speed, zero = none:
                             * center(t) = center + t*speed, t = Ray::time in [0,1))  objects/sphere.rs:45-51,69-91 */
    NRRT_OBJ_QUAD = 1,      /* v[0..2]=p v[3..5]=u v[6..8]=v    objects/plane.rs:95-127   */
    NRRT_OBJ_TRIANGLE = 2,  /* same as quad, Shape::Triangle                              */
    NRRT_OBJ_GROUP = 3,     /* BVH::from(children)  (Group, Scene, and the scene list)    */
    NRRT_OBJ_TRANSLATE = 4, /* v[0..2]=offset, one child        objects/translate.rs      */
    NRRT_OBJ_ROTATE_X = 5,  /* v[0]=angle (radians), one child  objects/rotate.rs:47-62   */
    NRRT_OBJ_ROTATE_Y = 6,
    NRRT_OBJ_ROTATE_Z = 7,
    NRRT_OBJ_SCALE = 8      /* v[0..2]=scale vector, one child  objects/scale.rs:44-58    */
};

typedef struct nrrt_object {
    uint32_t kind;        /* nrrt_obj_kind */
    uint32_t material;    /* index into materials (primitives only) */
    uint32_t first_child; /* index into nrrt_graph_desc.child_ids */
    uint32_t n_children;  /* groups: any; wrappers: 1; primitives: 0 */
    double v[9];
} nrrt_object;

enum nrrt_material_kind {
    NRRT_MAT_LAMBERTIAN = 0,    /* materials/lambertian.rs:39-55                    */
    NRRT_MAT_METAL = 1,         /* param = fuzz        materials/metal.rs:73-91     */
    NRRT_MAT_DIELECTRIC = 2,    /* param = ior         materials/dielectric.rs:39-67 */
    NRRT_MAT_DIFFUSE_LIGHT = 3  /* param = intensity   materials/diffuse_light.rs:63-75 */
};

typedef struct nrrt_material {
    uint32_t kind;
    uint32_t texture; /* index into textures (ignored by dielectric) */
    double param;
} nrrt_material;

enum nrrt_texture_kind {
    NRRT_TEX_SOLID = 0,   /* color                                   textures/solid_color.rs */
    NRRT_TEX_CHECKER = 1, /* a=even texture, b=odd texture, f0=scale textures/checker.rs:77-89 */
    NRRT_TEX_IMAGE = 2,   /* a=image index                           textures/image.rs:30-40 */
    NRRT_TEX_NOISE = 3,   /* |Fbm<Perlin>|: seed, octaves, f0=frequency, f1=lacunarity,
                             f2=persistence                          textures/noise.rs:79-145 */
    NRRT_TEX_MARBLE = 4   /* seed, f0=frequency (7 octaves)          textures/marble.rs:46-97 */
};

typedef struct nrrt_texture {
    uint32_t kind;
    uint32_t a, b;
    uint32_t seed;
    uint32_t octaves;
    uint32_t _pad;
    double color[3];
    double f0, f1, f2;
} nrrt_texture;

/* Decoded 8-bit RGB image, row-major, 3 bytes per texel, row 0 = top.
 * The reference converts with into_rgb32f() = u8/255 as f32 (textures/image.rs:24). */
typedef struct nrrt_image {
    uint32_t width, height;
    const uint8_t* rgb;
} nrrt_image;

typedef struct nrrt_graph_desc {
    uint32_t n_objects;
    const nrrt_object* objects;
    uint32_t n_child_ids;
    const uint32_t* child_ids;
    uint32_t n_materials;
    const nrrt_material* materials;
    uint32_t n_textures;
    const nrrt_texture* textures;
    uint32_t n_images;
    const nrrt_image* images;
    uint32_t root; /* object index of the scene list (a GROUP): Scene.objects = BVH::from(list) */
} nrrt_graph_desc;

/* CameraBuilder fields (camera.rs:30-41); angles in RADIANS (the CLI converts
 * degrees at cli.rs:369-379 before they reach the builder). */
typedef struct nrrt_camera_config {
    uint32_t width, height;
    uint32_t samples_per_pixel, ray_max_bounces;
    double background[3];
    double look_from[3], look_at[3], view_up[3];
    double defocus_angle, focus_dist, field_of_view;
} nrrt_camera_config;

/* The built Camera (camera.rs:206-227): what the kernels consume. */
typedef struct nrrt_camera {
    uint32_t width, height;
    uint32_t samples_per_pixel, ray_max_bounces;
    double background[3];
    double look_from[3];
    double defocus_disk_u[3], defocus_disk_v[3];
    double pixel_delta_u[3], pixel_delta_v[3];
    double viewport_top_left[3];
} nrrt_camera;

/* ======================================================================== */
/* 2. flat layer: device layout                                             */
/* ======================================================================== */

/* Node/child reference: bits 31..29 = type, bits 28..0 = index. */
#define NRRT_REF_TYPE_SHIFT 29u
#define NRRT_REF_INDEX_MASK 0x1FFFFFFFu
enum nrrt_ref_type {
    NRRT_REF_NODE = 0,     /* inner node: index into nodes/boxes        */
    NRRT_REF_SPHERE = 1,   /* index into sphere arrays                  */
    NRRT_REF_PLANE = 2,    /* index into plane arrays (quad + triangle) */
    NRRT_REF_INSTANCE = 3, /* index into instances                      */
    NRRT_REF_EMPTY = 7     /* BVH::Leaf(None)                           */
};
#define NRRT_REF(type, idx) ((((uint32_t)(type)) << NRRT_REF_TYPE_SHIFT) | ((uint32_t)(idx)))
#define NRRT_REF_TYPE(r) ((r) >> NRRT_REF_TYPE_SHIFT)
#define NRRT_REF_INDEX(r) ((r) & NRRT_REF_INDEX_MASK)
#define NRRT_REF_NONE 0xFFFFFFFFu /* == NRRT_REF(EMPTY, all ones) */

/* 64-byte traversal node: both children's boxes in f32 (nearest-rounded from
 * the f64 boxes; the kernel's certainty margins cover the rounding) and both
 * child references.  One 128-byte line holds two nodes; loaded as 4 x LDG.128. */
typedef struct nrrt_node {
    float lo[2][3]; /* lo[child][axis] */
    float hi[2][3];
    uint32_t child[2];
    uint32_t _pad[2];
} nrrt_node;

/* Exact f64 box (aabb.rs:6-11) used when the f32 test is inconclusive. */
typedef struct nrrt_box {
    double lo[3];
    double hi[3];
} nrrt_box;

/* 128-byte four-slot traversal node (one cache line, 8 x LDG.128): the binary tree above with every other level
 * folded away.  A wide node stands for one binary node B; its slots hold B's grandchildren in depth-first order
 * (or, where a child of B is a leaf, that child), so the leaves, their depth-first order and therefore every
 * tie-break (object.rs:110-114) are those of the binary tree, while a ray makes half as many dependent fetches.
 * What the reference tests on the way to a slot is kept exactly:
 *   - a slot that is an inner node must pass its own box test (object.rs:102);
 *   - a slot whose binary parent was folded away ("gated", meta bit 0) additionally needs that parent's box test
 *     to pass.  The parent's box encloses the slot's box and the slab test is monotone under IEEE rounding, so a
 *     slot box that certainly passes implies the gate passes; only inconclusive slots evaluate the gate in f64.
 * Leaves are not box-tested by the reference (object.rs:95-97): their slot box only culls what certainly misses. */
typedef struct nrrt_wnode {
    float lo[3][4];    /* lo[axis][slot], nearest-rounded from the f64 boxes */
    float hi[3][4];
    uint32_t child[4]; /* ref per slot (wide-node index for NODE refs); NRRT_REF_NONE = unused slot */
    uint32_t meta[4];  /* bit 0: gated slot */
} nrrt_wnode;
#define NRRT_WNODE_GATED 1u

/* One wrapper of an instance chain, outermost first. */
enum nrrt_xform_kind { NRRT_XF_TRANSLATE = 0, NRRT_XF_ROTATE = 1, NRRT_XF_SCALE = 2 };
typedef struct nrrt_xform {
    uint32_t kind;
    uint32_t _pad;
    /* TRANSLATE: to_obj[0..2] = offset.
     * ROTATE:    to_obj = rotation_mat  (3 columns, DMat3::from_axis_angle(axis,-angle)),
     *            to_world = rotation_mat_inv (rotate.rs:52-53).
     * SCALE:     to_obj = scale_matrix_inv columns x,y,z,w (xyz parts, 12 doubles),
     *            to_world = scale_matrix columns x,y,z,w (scale.rs:48-49). */
    double to_obj[12];
    double to_world[12];
} nrrt_xform;

typedef struct nrrt_instance {
    uint32_t first_xform; /* index into xforms, outermost wrapper first */
    uint32_t n_xforms;
    uint32_t inner;       /* ref of the wrapped object (node / sphere / plane / empty) */
    uint32_t _pad;
    nrrt_box inner_box;   /* bbox of `inner` when it is a NODE (tested on entry, object.rs:102) */
} nrrt_instance;

/* Instances nest (a wrapped group may contain wrappers again); a hit carries the
 * chain of instance indices from the top-level BVH down to the primitive. */
#define NRRT_MAX_INSTANCE_DEPTH 4

typedef struct nrrt_scene_desc {
    uint32_t abi_version;

    /* BVH */
    uint32_t n_nodes;
    const nrrt_node* nodes;      /* [n_nodes]                                   */
    const nrrt_box* child_boxes; /* [2*n_nodes] exact box of child c of node i at 2*i+c */
    uint32_t root;               /* ref of Scene.objects                        */
    nrrt_box root_box;           /* its bbox when root is a NODE                */

    /* spheres: one 32-byte record per sphere = {center.x, center.y, center.z, radius} (2 x LDG.128) */
    uint32_t n_spheres;
    const double* sphere_rec;      /* [n][4] */
    const uint32_t* sphere_material;
    const uint32_t* sphere_order;  /* DFS leaf order (tie-break, object.rs:110-114) */
    const uint32_t* sphere_object; /* graph object index (reported in nrrt_hit.object) */

    /* planes: one 128-byte record (= one cache line, 8 x LDG.128) per plane, everything Plane::hit reads, with
     * normal, d, w derived exactly as PlaneBuilder::build does (plane.rs:109-114):
     *   [0..2] normal  [3] d  [4..6] p  [7..9] w  [10..12] u  [13..15] v */
    uint32_t n_planes;
    const double* plane_rec;        /* [n][16] */
    const uint32_t* plane_material; /* bit 31 set = Triangle, else Quad */
    const uint32_t* plane_order;
    const uint32_t* plane_object;

    /* instances */
    uint32_t n_instances;
    const nrrt_instance* instances;
    const uint32_t* instance_order;
    uint32_t n_xforms;
    const nrrt_xform* xforms;

    /* shading tables */
    uint32_t n_materials;
    const nrrt_material* materials;
    uint32_t n_textures;
    const nrrt_texture* textures;
    uint32_t n_images;
    const nrrt_image* images;

    uint32_t max_stack; /* worst-case traversal stack entries over the four-slot nodes (validated by the host) */

    /* moving spheres (sphere.rs:110-111): speed vector per sphere, or NULL when no sphere moves (every shipped
     * scene); kept out of sphere_rec so static scenes keep the 32-byte record */
    const double* sphere_speed; /* [n][3] or NULL */

    /* Four-slot traversal nodes: what the kernels walk (nodes / child_boxes above describe the same trees in binary
     * form and stay on the host).  wide_boxes[8*i + 2*s] = exact box of slot s of wide node i (inner-node slots),
     * wide_boxes[8*i + 2*s + 1] = exact box of its folded-away binary parent (gated slots). */
    uint32_t n_wnodes;
    const nrrt_wnode* wnodes;            /* [n_wnodes] */
    const nrrt_box* wide_boxes;          /* [8*n_wnodes] */
    uint32_t wide_root;                  /* `root` as a wide ref */
    const uint32_t* instance_wide_inner; /* [n_instances]: instances[i].inner as a wide ref */
} nrrt_scene_desc;

#define NRRT_PLANE_TRIANGLE_BIT 0x80000000u

/* ---- host side: reference's BVH build + flatten (no GPU needed) -------- */
typedef struct nrrt_host_scene nrrt_host_scene;

/* Builds the object graph, runs BVH::from exactly as the reference does and
 * flattens it.  `graph` is borrowed for the call only.  Returns NULL on error
 * (message via nrrt_host_last_error). */
nrrt_host_scene* nrrt_host_build(const nrrt_graph_desc* graph);

/* Same, with build options.  NRRT_BUILD_REFERENCE (0) is nrrt_host_build: the reference's tree, node for node.
 * NRRT_BUILD_SAH replaces the inner nodes of every BVH::from tree by a binned surface-area-heuristic build
 * (opt-in: the reference's median-split tree costs roughly twice the node visits on meshes).  Leaves, records
 * and the depth-first leaf order that decides equal-t ties (object.rs:110-114) stay the reference's, so hits
 * are the reference's except where a ray grazes a bounding box within f64 rounding: there the reference's
 * result depends on which inner boxes its own tree tests (object.rs:102), and only the reference tree
 * reproduces that. */
enum { NRRT_BUILD_REFERENCE = 0, NRRT_BUILD_SAH = 1 };
nrrt_host_scene* nrrt_host_build_ex(const nrrt_graph_desc* graph, uint32_t flags);
const nrrt_scene_desc* nrrt_host_scene_desc(const nrrt_host_scene* scene);
void nrrt_host_free(nrrt_host_scene* scene);
const char* nrrt_host_last_error(void);

/* CameraBuilder::build (camera.rs:94-159). */
int nrrt_host_camera_build(const nrrt_camera_config* config, nrrt_camera* out);

/* ---- host side: native scene loader (SURVEY.md §8(f) N1) ---------------- */
/* Mirror of the CLI's CameraConfig (cli.rs:157-270): every field optional; `present` says which were given.
 * Angles in DEGREES here, like the CLI flags and the scene files (converted by nrrt_camera_file_to_config). */
enum {
    NRRT_CAM_WIDTH = 1 << 0, NRRT_CAM_HEIGHT = 1 << 1, NRRT_CAM_ASPECT_RATIO = 1 << 2, NRRT_CAM_BACKGROUND = 1 << 3,
    NRRT_CAM_LOOK_AT = 1 << 4, NRRT_CAM_LOOK_FROM = 1 << 5, NRRT_CAM_VIEW_UP = 1 << 6, NRRT_CAM_FOV = 1 << 7,
    NRRT_CAM_DEFOCUS = 1 << 8, NRRT_CAM_FOCUS = 1 << 9, NRRT_CAM_SPP = 1 << 10, NRRT_CAM_BOUNCES = 1 << 11
};
typedef struct nrrt_camera_file {
    uint32_t present;
    uint32_t width, height, samples_per_pixel, ray_max_bounces;
    uint32_t _pad;
    double aspect_ratio;
    double background[3], look_at[3], look_from[3], view_up[3];
    double field_of_view_deg, defocus_angle_deg, focus_distance;
} nrrt_camera_file;

typedef struct nrrt_loaded_scene nrrt_loaded_scene;
/* SceneConfig::try_load_scene + try_build's object graph (scene_config.rs:411-492): .json / .toml by extension;
 * paths inside the file (Image.path, Scene.path) resolve against base_dir (NULL = process CWD, like the
 * reference).  JPEG textures are decoded natively (baseline).  NULL on error (nrrt_load_last_error). */
nrrt_loaded_scene* nrrt_load_scene(const char* path, const char* base_dir);
const nrrt_graph_desc* nrrt_loaded_graph(const nrrt_loaded_scene* scene); /* feed to nrrt_host_build */
int nrrt_loaded_camera(const nrrt_loaded_scene* scene, nrrt_camera_file* out); /* the file's [camera] section */
void nrrt_loaded_free(nrrt_loaded_scene* scene);
const char* nrrt_load_last_error(void);
/* CameraConfig::merge_with (cli.rs:316-355) and try_update onto CameraBuilder::default() (cli.rs:357-402). */
void nrrt_camera_file_merge(nrrt_camera_file* base, const nrrt_camera_file* over);
int nrrt_camera_file_to_config(const nrrt_camera_file* file, nrrt_camera_config* out);

/* ---- device side -------------------------------------------------------- */
typedef struct nrrt_ctx nrrt_ctx;

/* One context per GPU (one process per GPU under torch.distributed). */
int nrrt_create(int device, nrrt_ctx** out);
void nrrt_destroy(nrrt_ctx* ctx);
const char* nrrt_last_error(const nrrt_ctx* ctx); /* ctx may be NULL: last create error */

/* Launch on this CUDA stream (a cudaStream_t passed as void*); default 0. */
int nrrt_set_stream(nrrt_ctx* ctx, void* cuda_stream);

/* Copies the flat scene to HBM (host pointers borrowed for the call only). */
int nrrt_scene_upload(nrrt_ctx* ctx, const nrrt_scene_desc* scene);

/* Closest-hit query result = HitRecord (hitable.rs:15-22) + ids. */
typedef struct nrrt_hit {
    double t;          /* +inf on miss */
    double point[3];
    double normal[3];
    double uv[2];
    uint32_t prim;     /* winning primitive ref (NRRT_REF_NONE on miss) */
    uint32_t material;
    uint32_t front_face;
    uint32_t object;   /* graph object index of the winning primitive (0xFFFFFFFF on miss) */
    uint32_t depth;    /* number of instance levels above the primitive */
    uint32_t inst[NRRT_MAX_INSTANCE_DEPTH]; /* instance indices, outermost first */
    uint32_t _pad;
} nrrt_hit;

typedef struct nrrt_hit_compact {
    double t;      /* +inf on miss */
    uint32_t prim; /* winning primitive ref (NRRT_REF_NONE on miss) */
    uint32_t depth_inst0; /* instance levels above the primitive | outermost instance index << 3 */
} nrrt_hit_compact;

enum {
    NRRT_TRACE_ORDERED = 0,    /* near-first traversal with conservative t-shrinking (render path) */
    NRRT_TRACE_VISIT_ALL = 1,  /* visit exactly the reference's node set (no shrinking)            */
    NRRT_TRACE_HOST_BUFFERS = 0,
    NRRT_TRACE_DEVICE_BUFFERS = 2,
    NRRT_TRACE_COUNT = 4,      /* also fill node_visits / box_exact / prim_tests (per-ray atomics: slower) */
    NRRT_TRACE_COMPACT = 8     /* `out` is n x nrrt_hit_compact (16 bytes per ray: t and the winning primitive) instead of
                                  n x nrrt_hit: the closest-hit query alone, no HitRecord — the traversal-only
                                  microbenchmark that bench.py reports the render kernels against */
};

typedef struct nrrt_trace_stats {
    uint64_t node_visits;   /* NRRT_TRACE_COUNT: inner nodes fetched                 */
    uint64_t box_exact;     /*   f32-inconclusive box tests redone in f64            */
    uint64_t prim_tests;    /*   exact primitive tests                               */
    double kernel_ms;       /* CUDA-event time of the kernel (always)                */
} nrrt_trace_stats;

/* Ray::time (ray.rs:8) of the rays given to nrrt_trace_rays, default 0.  Only moving spheres read it. */
int nrrt_set_trace_time(nrrt_ctx* ctx, double time);

/* BVH::hit (object.rs:89-121) for n rays: rays = n x {ox,oy,oz,dx,dy,dz}. */
int nrrt_trace_rays(nrrt_ctx* ctx, const double* rays, uint64_t n, double tmin, double tmax,
                    uint32_t flags, nrrt_hit* out, nrrt_trace_stats* stats /* may be NULL */);

enum nrrt_render_mode {
    NRRT_MODE_WAVEFRONT = 0, /* raygen / extend / shade+compact kernels over ray queues */
    NRRT_MODE_MEGAKERNEL = 1, /* one kernel, per-thread path loop, whole state in registers */
    NRRT_MODE_FUSED = 2,      /* persistent warps: traverse with warp-voted in-place shading, path state in
                                 shared memory (no ray / hit-record round trips through HBM)   */
    NRRT_MODE_POOL = 3,       /* persistent warps, each scheduling a pool of path slots held in shared memory:
                                 node / primitive / instance / shade stages run on whichever slots are ready,
                                 so every stage runs with (nearly) all 32 lanes                  */
    NRRT_MODE_AUTO = 4        /* the product path: POOL for scenes with deep trees (meshes), FUSED otherwise —
                                 whichever measured faster on B200 for that kind of scene; nrrt_render_stats.mode
                                 reports the design that ran.  All designs give the bit-identical image. */
};

typedef struct nrrt_render_opts {
    uint64_t seed;        /* Philox key; the reference seeds ChaCha8 with 0 (camera.rs:318) */
    uint32_t mode;        /* nrrt_render_mode */
    uint32_t rank, world; /* tile partition: this context renders row-blocks b with b % world == rank */
    uint32_t rows_per_block; /* height of one row-block (0 -> default 8) */
    uint32_t max_slots;   /* wavefront: path slots in flight (0 -> auto) */
    uint32_t flags;       /* NRRT_RENDER_* */
} nrrt_render_opts;

enum {
    NRRT_RENDER_OUT_HOST = 0,
    NRRT_RENDER_OUT_DEVICE = 1, /* out_rgb is a device pointer */
    NRRT_RENDER_COUNT = 2,      /* instrumented megakernel: also count node visits / primitive tests (slower) */
    NRRT_RENDER_OUT_PACKED = 4  /* out_rgb holds only the rows this rank owns, packed in ascending row order
                                   (stats.pixels * 3 floats): what a multi-GPU gather sends, without a pack step */
};

typedef struct nrrt_render_stats {
    uint64_t paths;        /* pixel samples traced by this context             */
    uint64_t segments;     /* closest-hit queries issued (camera.rs:280)       */
    uint64_t launches;     /* kernels launched                                 */
    double device_ms;      /* CUDA-event time, first launch -> last launch     */
    double extend_ms;      /* share of device_ms in the traverse/intersect kernel (wavefront) */
    uint64_t extend_launches;
    uint32_t pixels;       /* pixels owned by this rank                        */
    uint32_t mode;         /* nrrt_render_mode that ran (resolves NRRT_MODE_AUTO) */
    uint64_t node_visits;  /* NRRT_RENDER_COUNT only: inner nodes fetched      */
    uint64_t box_exact;    /*   f32-inconclusive / root box tests done in f64  */
    uint64_t prim_tests;   /*   exact primitive tests                          */
    uint64_t inst_entries; /*   wrapper chains applied to a ray (instance leaves reached) */
    uint64_t inst_misses;  /*   ... of which the nested root box was missed    */
} nrrt_render_stats;

typedef void (*nrrt_progress_fn)(uint64_t pixels_done, uint64_t pixels_total, void* user);

/* Camera::render (camera.rs:302-343).  out_rgb: width*height*3 f32, row-major
 * interleaved RGB, linear radiance (no gamma, no clamp).  With world > 1 only
 * the rows owned by `rank` are written (others left untouched). */
int nrrt_render(nrrt_ctx* ctx, const nrrt_camera* camera, const nrrt_render_opts* opts,
                float* out_rgb, nrrt_progress_fn progress, void* user, nrrt_render_stats* stats);

/* Camera::render over several GPUs of one box from ONE process (what `nr-ray-tracer render --gpus N` calls; the
 * one-process-per-GPU form with torch.distributed / NCCL is nr_ray_tracer_b200/distributed.py).  One host thread and
 * one context per device: every device uploads the scene, renders the rows r with r % n_devices == its index
 * end to end (same Philox streams, so the image is bit-identical to a single-GPU render) and the rows are brought
 * together inside the library:
 *   - host out_rgb (default): each device copies its rows straight into the caller's image with one strided D2H
 *     copy, all devices in parallel over their own PCIe links;
 *   - NRRT_RENDER_OUT_DEVICE: out_rgb is memory of devices[0]; the other devices render packed rows, push them to
 *     devices[0] with peer-to-peer copies over NVLink and one kernel there places them.
 * opts->rank / world / rows_per_block are ignored (set per device).  stats (may be NULL): paths, segments, launches
 * and pixels summed over the devices, device_ms = the slowest device.  progress (may be NULL) is called under a lock
 * with the pixels finished on all devices.  err (may be NULL) receives the message of the first failing device. */
int nrrt_render_multi(const int* devices, int n_devices, const nrrt_scene_desc* scene, const nrrt_camera* camera,
                      const nrrt_render_opts* opts, float* out_rgb, nrrt_progress_fn progress, void* user,
                      nrrt_render_stats* stats, char* err, size_t err_len);

/* Output stage (§8(f) N2): gamma_correction (image.rs:53-57: p.powf(gamma) per channel, f32) followed by
 * DynamicImage::to_rgb8 (render.rs:85-86: clamp to [0,1], x255, round) on the GPU, so only W*H*3 bytes cross PCIe.
 * `rgb` is W*H*3 f32 (device pointer if NRRT_RENDER_OUT_DEVICE is set in flags, else host); `out_rgb8` is a
 * caller-owned HOST buffer of W*H*3 bytes. */
int nrrt_encode_rgb8(nrrt_ctx* ctx, const float* rgb, uint32_t width, uint32_t height, float gamma, uint32_t flags,
                     uint8_t* out_rgb8);

/* The work items of a pixel: a render sums a pixel's samples chunk by chunk, and the chunks depend only on spp and the
 * size of the whole image (never on the partition, so an N-GPU image is the 1-GPU image bit for bit).  Writes the first
 * sample of every chunk and spp as the last entry (n_chunks + 1 values, at most `max`); returns n_chunks. */
uint32_t nrrt_chunk_starts(uint32_t samples_per_pixel, uint64_t total_pixels, uint32_t* starts, uint32_t max);

/* The work items of one rank's render, decoded by the functions the kernels use (nrrt_device.cu decode_item /
 * owned_pixel): items [first, first + n) as 4 values each — x, y, first sample, one past the last sample — in the
 * order they are handed out (chunk-major; inside a chunk the rank's pixels in strips of up to 8 rows, column by column).
 * Returns the number of items of that render (owned pixels x chunks), 0 for arguments nrrt_render would refuse.
 * For tests and bindings: every (owned pixel, sample) must appear exactly once, whatever the partition. */
uint32_t nrrt_work_items(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank, uint32_t world,
                         uint32_t rows_per_block, uint32_t first, uint32_t n, uint32_t* out);

/* The same for one pass of a progressive render: the work items of chunks [c0, c1) (c1 clamped to n_chunks), numbered
 * from 0 in the order that pass hands them out.  nrrt_work_items is c0 = 0, c1 = all.  Returns 0 also when c0 > n_chunks. */
uint32_t nrrt_pass_items(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank, uint32_t world,
                         uint32_t rows_per_block, uint32_t c0, uint32_t c1, uint32_t first, uint32_t n, uint32_t* out);

/* ---- progressive rendering ---------------------------------------------------------------------------------------
 * One frame rendered in passes on one context.  A pass renders the next whole chunks of every owned pixel (pass
 * boundaries are nrrt_chunk_starts boundaries) and adds their partial sums, in chunk order, into a per-pixel f64 sum the
 * handle keeps in device memory (24 B per owned pixel, owned rows packed: row j, column x, RGB).  A pixel's sample s
 * traces the same path in whichever pass it runs, so:
 *   - after the last pass the image is nrrt_render's, bit for bit, whatever the passes were;
 *   - after samples [0, s) the image is the sum over those chunks divided by s (the CPU oracle's render_chunked);
 *   - a pass needs scratch for its own chunks only (24 B per owned pixel and chunk).
 * camera->samples_per_pixel, opts->seed / mode / rank / world / rows_per_block / max_slots are fixed at creation; the
 * output flags of opts are ignored (nrrt_accum_image takes them), NRRT_RENDER_COUNT is honoured.  Every call fails with
 * NRRT_ERR_NO_SCENE once nrrt_scene_upload has replaced the context's scene.  Error messages: nrrt_last_error(ctx).
 * Free the handle before its context. */
typedef struct nrrt_accum nrrt_accum;
int nrrt_accum_create(nrrt_ctx* ctx, const nrrt_camera* camera, const nrrt_render_opts* opts, nrrt_accum** out);
/* Renders the next whole chunks until at least min(min_samples, spp) samples per pixel are done (nothing if they are
 * already; stats are then zero but for pixels).  stats (may be NULL) describe this pass. */
int nrrt_accum_render(nrrt_accum* accum, uint32_t min_samples, nrrt_render_stats* stats);
/* Samples per pixel done so far (a chunk boundary; spp when the frame is complete). */
uint32_t nrrt_accum_samples(const nrrt_accum* accum);
/* The image so far: sums / samples done, as f32, laid out as nrrt_render lays out out_rgb (flags
 * NRRT_RENDER_OUT_DEVICE / NRRT_RENDER_OUT_PACKED as there).  NRRT_ERR_INVALID before the first pass. */
int nrrt_accum_image(nrrt_accum* accum, float* out_rgb, uint32_t flags);
/* Host copy of the sums (stats.pixels x 3 f64, owned rows packed) and the samples they hold, e.g. to resume later. */
int nrrt_accum_save(const nrrt_accum* accum, double* sums, uint32_t* samples_done);
/* Loads what nrrt_accum_save wrote, into an accumulator of the same frame (camera, opts, scene), possibly on another
 * context.  NRRT_ERR_INVALID if samples_done is not a chunk boundary of the frame (so also above spp). */
int nrrt_accum_restore(nrrt_accum* accum, const double* sums, uint32_t samples_done);
void nrrt_accum_free(nrrt_accum* accum);

/* ---- adaptive sampling -------------------------------------------------------------------------------------------
 * An adaptive frame is a progressive frame created with tolerances.  Its passes render the next whole chunks, as
 * above, but only for the pixels still ACTIVE.  After a pass every pixel that took part is tested; a pixel that passes
 * the test is RETIRED: its sum, second moment and sample count never change again.  Per owned pixel the handle keeps
 *   S  the f64 RGB sum of its samples (as above),
 *   Q  the f64 RGB sum over its chunks of P_c * P_c / n_c (P_c: chunk c's partial sum, n_c: its sample count), added in
 *      chunk order by the thread that adds P_c to S, without FMA contraction: Q = Q + (p * p) / n_c, each step rounded,
 *   N  its sample count (a nrrt_chunk_starts boundary) and K its chunk count.
 * The test (nrrt_adaptive_converged), evaluated in f64 per channel in this order:
 *   m = S / N;  d = max(Q - (S * S) / N, 0);  e2 = d / ((K - 1) * N);  tol = abs_error + rel_error * |m|
 * e2 is the squared standard error of the mean estimated from the chunks as batch means (E[sum n_c (m_c - m)^2] =
 * (K - 1) sigma^2 holds for unequal batches too).  A pixel is converged iff K >= 2, N >= min_samples, a tolerance is
 * positive, and e2 <= tol * tol in all three channels (NaN compares false).  Tolerance 0 therefore never retires a
 * pixel: such a frame is nrrt_render's image bit for bit.
 * A pixel's value is S / N as f32: the CPU oracle's render_chunked over the chunks it received, bit for bit.  Decisions
 * are made at pass ends only, so the result depends on the scene, camera, seed, tolerances and pass schedule, and not on
 * the kernel design, slot count or partition.  On an adaptive handle:
 *   - nrrt_accum_render renders the active pixels' next chunks up to min_samples, then tests them; its stats count
 *     what ran (stats.pixels = the active pixels of the pass);
 *   - nrrt_accum_samples is the frame's chunk boundary: retired pixels sit below it;
 *   - nrrt_accum_image divides each pixel by its own N;
 *   - nrrt_accum_save / _restore fail with NRRT_ERR_INVALID (use the _adaptive_ pair). */
typedef struct nrrt_adaptive_opts {
    double rel_error, abs_error; /* >= 0 and finite, else NRRT_ERR_INVALID */
    uint32_t min_samples;        /* a pixel is tested only from this many samples (and two chunks) on */
    uint32_t _pad;
} nrrt_adaptive_opts;
int nrrt_accum_create_adaptive(nrrt_ctx* ctx, const nrrt_camera* camera, const nrrt_render_opts* opts,
                               const nrrt_adaptive_opts* adaptive, nrrt_accum** out);
/* Pixels of this rank still active (0 = frame finished; every owned pixel before the first pass).  0 for a handle
 * that is not adaptive. */
uint32_t nrrt_accum_active(const nrrt_accum* accum);
/* N per pixel (u32), laid out as nrrt_accum_image lays out one channel (flags NRRT_RENDER_OUT_DEVICE / _PACKED). */
int nrrt_accum_sample_map(nrrt_accum* accum, uint32_t* out, uint32_t flags);
/* sqrt(e2) per channel as f32 (+inf where K < 2), laid out as nrrt_accum_image. */
int nrrt_accum_error_image(nrrt_accum* accum, float* out_rgb, uint32_t flags);
/* Host copy of S, Q (stats.pixels x 3 f64 each) and N (stats.pixels u32), owned rows packed. */
int nrrt_accum_adaptive_save(const nrrt_accum* accum, double* sums, double* sumsq, uint32_t* samples);
/* Loads what nrrt_accum_adaptive_save wrote into an adaptive handle of the same frame.  Every N must be a chunk
 * boundary of the frame, at least one chunk, and one value below the largest N only for a pixel that passes the test
 * (a retired pixel); the active set is rebuilt by re-evaluating the test.  NRRT_ERR_INVALID otherwise. */
int nrrt_accum_adaptive_restore(nrrt_accum* accum, const double* sums, const double* sumsq, const uint32_t* samples);
/* The test above on one pixel's state (1 = converged).  For tests and bindings. */
int nrrt_adaptive_converged(const double S[3], const double Q[3], uint32_t samples, uint32_t chunks,
                            const nrrt_adaptive_opts* adaptive);
/* nrrt_pass_items for a pass over the owned pixels active[0 .. n_active) only (owned-pixel indices in the order
 * nrrt_pass_items visits a chunk's pixels, strictly ascending, each below the owned pixel count): inside each chunk the
 * items follow the list.  Returns the number of items, 0 also for a list that breaks those rules. */
uint32_t nrrt_pass_items_active(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank,
                                uint32_t world, uint32_t rows_per_block, uint32_t c0, uint32_t c1,
                                const uint32_t* active, uint32_t n_active, uint32_t first, uint32_t n, uint32_t* out);

/* ---- denoising ---------------------------------------------------------------------------------------------------
 * An extra output of a frame, like nrrt_accum_error_image: the frame's own image, state and kernels are untouched.
 *
 * Guides (AOVs).  Per owned pixel, the mean over its samples s = 0 .. n-1 of the first hit of sample s's camera ray (the
 * render's ray: same Philox counters, so the same jitter, lens point and shutter time), traced on [0.001, inf):
 *   normal = the hit record's normal (the one shading sees; quirk Q4: a Scale wrapper leaves it in object space),
 *   albedo = the material texture's colour at the hit (Lambertian, Metal), (1, 1, 1) (Dielectric), the texture colour
 *            clamped to [0, 1] per channel (DiffuseLight);
 *   a miss gives normal (0, 0, 0) and albedo = the background clamped to [0, 1].
 * Summed in f64 in sample order, divided by n, cast to f32: the CPU oracle's restatement (tests/aov_ref.py) bit for bit.
 *
 * Filter.  An edge-avoiding a-trous wavelet filter (SVGF form) on the albedo-demodulated image, guided by the normals,
 * the albedo and the frame's per-pixel error estimate.  Every f32 operation is rounded on its own (no FMA), in this
 * order.  Per pixel p:  C = (float)(S / N);  e2 = (float)e2 of the adaptive test, +inf where K < 2;  A, Nrm the guides.
 *   prologue:   a = max(A, 2^-8) per channel;  E = C / a;  v = ((e2_r/(a_r*a_r) + e2_g/(a_g*a_g)) + e2_b/(a_b*a_b)) * (1/9)
 *   iteration i = 0 .. iterations-1, h = 2^i, from (E, v) of the previous one:
 *     l = ((E_r + E_g) + E_b) / 3;   sums Sw = SE = Sv = 0;
 *     taps q = p + h*(dx, dy), dy outer and dx inner over -2..2, taps outside the image skipped;
 *     k = b[|dx|] * b[|dy|], b = {3/8, 1/4, 1/16};
 *     centre tap: w = k;  other taps: w = ((k * wn) * wa) * wc with
 *       wn = max(Nrm_p . Nrm_q, 0) squared 7 times (dot products (x*x' + y*y') + z*z'),
 *       wa = 1 / (1 + |A_p - A_q|^2 * 64),
 *       wc = 1 where v_p = +inf, else 1 / (1 + (l_p - l_q)^2 / (sigma_color^2 * v_p + 1e-10)), sigma_color^2 in f32;
 *       a tap with w * w == 0 adds nothing (w == 0, or w so small that w * w underflows: 0 * inf never reaches
 *       the sums; the centre's w * w = 81/4096);
 *     Sw += w;  SE_c += w * E_q,c;  Sv += (w * w) * v_q  (in tap order);   E' = SE / Sw;  v' = Sv / (Sw * Sw)
 *   epilogue:   out = E' * a per channel.
 * Sw >= 9/64 (the centre tap), so nothing divides by zero. */
typedef struct nrrt_denoise_opts {
    uint32_t iterations;  /* 1..8; 0 -> 5 */
    uint32_t aov_samples; /* guides over the first n samples, 1..spp; 0 -> min(spp, 16) */
    float sigma_color;    /* > 0 and finite; 0 -> 4 */
    uint32_t _pad;
} nrrt_denoise_opts;
/* The guides of the frame's first aov_samples samples per pixel (0: min(spp, 16)), f32 RGB each, laid out as
 * nrrt_accum_image lays out the image (flags NRRT_RENDER_OUT_DEVICE / _PACKED); either output may be NULL.  Works on any
 * handle, before the first pass too.  The handle computes them on first use for a given aov_samples and keeps them
 * (24 B per owned pixel, freed with the handle); passes never change them. */
int nrrt_accum_aov(nrrt_accum* accum, uint32_t aov_samples, float* albedo, float* normal, uint32_t flags);
/* The filter above on the frame so far, W x H x 3 f32 (NRRT_RENDER_OUT_DEVICE as in nrrt_accum_image; opts may be NULL:
 * every default).  NRRT_ERR_INVALID for a plain handle (no error estimate), world > 1 or NRRT_RENDER_OUT_PACKED (the
 * filter reads neighbours across rows), before the first pass, and for options out of range. */
int nrrt_accum_denoise(nrrt_accum* accum, const nrrt_denoise_opts* opts, float* out_rgb, uint32_t flags);

/* sizeof() of the ABI structs as compiled (which = 0..20: object, material, texture,
 * image, graph_desc, camera_config, camera, node, box, xform, instance, scene_desc, hit, trace_stats,
 * render_opts, render_stats, camera_file, wnode, hit_compact, adaptive_opts, denoise_opts) so a binding can verify its
 * mirror of this header. */
size_t nrrt_abi_sizeof(int which);

#ifdef __cplusplus
}
#endif
#endif /* NRRT_H */
