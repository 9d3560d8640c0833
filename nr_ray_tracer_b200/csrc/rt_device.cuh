// rt_device.cuh — device functions of the path-tracing hot path (sm_100a).
//
// Numerics contract (DESIGN.md "Exactness"):
//  * everything that decides hit/miss, the winning primitive or t is f64 in the reference's
//    operation order, written with __dadd_rn/__dmul_rn/__ddiv_rn/__dsqrt_rn so that nvcc can
//    never contract a*b+c into an FMA (rustc does not) while f32 code keeps FMA;
//  * f32 appears only in the box *filter*: a slab test on nearest-rounded f32 boxes with an
//    explicit error margin that classifies a box as certain-hit / certain-miss / inconclusive;
//    inconclusive inner nodes are re-tested with the reference's exact f64 slab test
//    (aabb.rs:110-132), so the set of primitives that get tested is the reference's set
//    restricted to those that can still win.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/nrrt.h"

#ifndef NRRT_LEAF_VOTE
#define NRRT_LEAF_VOTE 1   // 1: a warp serves one leaf kind per round (primitive tests OR instance entries)
#endif
#ifndef NRRT_HIT_SINK
#define NRRT_HIT_SINK 1    // 1: the wavefront traverse kernel hands hit attributes to the shade kernel
#endif
// Scene features a kernel instantiation has to handle.  nrrt_scene_upload computes the mask of the uploaded scene
// and the render path picks the tightest instantiation, so e.g. the Cornell box runs kernels without sphere,
// image, noise or dielectric code and spheres.toml runs kernels without any instance machinery.
#define NRRT_F_SPHERES 1u
#define NRRT_F_PLANES 2u
#define NRRT_F_INSTANCES 4u
#define NRRT_F_TEXTURED 8u      // any non-solid texture (checker / image / noise / marble)
#define NRRT_F_DIELECTRIC 16u
#define NRRT_F_MOTION 32u       // moving spheres (SphereBuilder::with_speed): rays carry Ray::time
#define NRRT_F_ALL 63u
// Not a scene feature: the launch is an adaptive pass and decodes its work items through RenderParams.active
// (decode_item<true>).  Plain renders launch instantiations without it.
#define NRRT_F_ACTIVE 64u
#ifndef NRRT_STACK_CAP
#define NRRT_STACK_CAP 32          // traversal stack entries per thread (host validates max_stack)
#endif
#define NRRT_REF_POP 0xC0000000u   // type 6: "leave instance level" marker on the stack
// Checked build (-DNRRT_CHECKED=1, tools/build_variant.py): every traversal-stack push, slot index and scene index the
// kernels form is bounds-checked on the device and a violation aborts the launch (printf + trap), so a test run of the
// checked library fails loudly.  The stand-in for compute-sanitizer memcheck, which is closed on the GPU pool.
#if defined(NRRT_CHECKED) && NRRT_CHECKED
#define NRRT_CHECK(cond, what)                                                                         \
    do {                                                                                               \
        if (!(cond)) {                                                                                 \
            printf("NRRT_CHECK failed: %s (%s:%d) block %d thread %d\n", what, __FILE__, __LINE__, (int)blockIdx.x, (int)threadIdx.x); \
            __trap();                                                                                  \
        }                                                                                              \
    } while (0)
#else
#define NRRT_CHECK(cond, what) do { } while (0)
#endif
#define NRRT_INF __longlong_as_double(0x7ff0000000000000LL)

// --------------------------------------------------------------------------- device scene
struct DevScene {
    const float4* wnodes;  // four-slot nodes (nrrt_wnode), 8 x float4 each
    const nrrt_box* wide_boxes;  // [8 * n]: own box / gate box per slot
    uint32_t root;         // wide ref
    // the same trees in binary form (nrrt_node), uploaded only for small scenes: a tree of a dozen nodes gains nothing
    // from folding levels, and the two-box visit is half the instructions of the four-box one
    const float4* bnodes;  // 4 x float4 per node, or nullptr
    const nrrt_box* bchild_boxes;
    const uint32_t* inst_binner;  // per instance: inner as a binary ref
    uint32_t broot;
    nrrt_box root_box;
    const double* sphere_rec;  // [n][4]: center xyz, radius
    const double* sphere_speed;  // [n][3] or nullptr when no sphere moves
    const uint32_t* sphere_material;
    const uint32_t* sphere_order;
    const uint32_t* sphere_object;
    const double* plane_rec;   // [n][16]: normal xyz, d, p xyz, w xyz, u xyz, v xyz (one 128-byte line)
    const float4* plane32;     // [n][4]: the f32 reject-only view of the same planes (plane_prereject), built at upload
    const uint32_t* plane_material;
    const uint32_t* plane_order;
    const uint32_t* plane_object;
    const nrrt_instance* instances;
    const uint32_t* instance_order;
    const nrrt_xform* xforms;
    const nrrt_material* materials;
    const nrrt_texture* textures;
    const uint8_t* material_flags;  // bit0: texture chain needs uv
    const cudaTextureObject_t* image_tex;
    const uint2* image_size;
    const uint8_t* perm;            // noise permutation tables, 256 B per (texture, octave)
    const uint32_t* perm_base;      // per texture: first table index
    uint32_t n_nodes, n_wnodes, n_spheres, n_planes, n_instances, n_materials, n_textures;
};

// --------------------------------------------------------------------------- exact f64 helpers
struct d3 {
    double x, y, z;
};
__device__ __forceinline__ d3 mk3(double x, double y, double z) { return d3{x, y, z}; }
__device__ __forceinline__ d3 ld3(const double* p) { return d3{p[0], p[1], p[2]}; }
__device__ __forceinline__ double xadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double xmul(double a, double b) { return __dmul_rn(a, b); }
// (measured on B200: out-of-line copies of the division / square root / Philox sequences shrink the kernels by 10 %
// but cost 5-15 % throughput — calls force live f64 state through the stack — so they stay inline)
#ifndef NRRT_DIV_INLINE
#define NRRT_DIV_INLINE __forceinline__
#endif
__device__ NRRT_DIV_INLINE double xdiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ NRRT_DIV_INLINE double xsqrt(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ d3 add3(d3 a, d3 b) { return d3{xadd(a.x, b.x), xadd(a.y, b.y), xadd(a.z, b.z)}; }
__device__ __forceinline__ d3 sub3(d3 a, d3 b) { return d3{xsub(a.x, b.x), xsub(a.y, b.y), xsub(a.z, b.z)}; }
__device__ __forceinline__ d3 neg3(d3 a) { return d3{-a.x, -a.y, -a.z}; }
__device__ __forceinline__ d3 scale3(d3 a, double s) { return d3{xmul(a.x, s), xmul(a.y, s), xmul(a.z, s)}; }
__device__ __forceinline__ d3 mul3(d3 a, d3 b) { return d3{xmul(a.x, b.x), xmul(a.y, b.y), xmul(a.z, b.z)}; }
__device__ __forceinline__ d3 div3(d3 a, double s) { return d3{xdiv(a.x, s), xdiv(a.y, s), xdiv(a.z, s)}; }
// glam dot: (x*x') + (y*y') + (z*z')
__device__ __forceinline__ double dot3(d3 a, d3 b) {
    return xadd(xadd(xmul(a.x, b.x), xmul(a.y, b.y)), xmul(a.z, b.z));
}
__device__ __forceinline__ d3 cross3(d3 a, d3 b) {
    return d3{xsub(xmul(a.y, b.z), xmul(b.y, a.z)), xsub(xmul(a.z, b.x), xmul(b.z, a.x)),
              xsub(xmul(a.x, b.y), xmul(b.x, a.y))};
}
// glam normalize: v * (1/sqrt(v.v))
__device__ __forceinline__ d3 normalize3(d3 a) { return scale3(a, xdiv(1.0, xsqrt(dot3(a, a)))); }
// ray.at(t) = origin + t*direction (ray.rs:40-42)
__device__ __forceinline__ d3 ray_at(d3 o, d3 d, double t) { return add3(o, scale3(d, t)); }
// Rust f64::signum
__device__ __forceinline__ double signum(double x) {
    if (x != x) return x;
    return (__double_as_longlong(x) < 0) ? -1.0 : 1.0;
}
// DMat3 * v : c0*v.x + c1*v.y + c2*v.z, left to right (m = 9 doubles, column major)
__device__ __forceinline__ d3 mat3_mul(const double* m, d3 v) {
    d3 r = scale3(ld3(m), v.x);
    r = add3(r, scale3(ld3(m + 3), v.y));
    r = add3(r, scale3(ld3(m + 6), v.z));
    return r;
}
// DMat4::transform_point3 / transform_vector3 on the xyz rows (m = 12 doubles: x,y,z,w columns)
__device__ __forceinline__ d3 mat4_point(const double* m, d3 v) {
    d3 r = scale3(ld3(m), v.x);
    r = add3(scale3(ld3(m + 3), v.y), r);
    r = add3(scale3(ld3(m + 6), v.z), r);
    r = add3(ld3(m + 9), r);
    return r;
}
__device__ __forceinline__ d3 mat4_vector(const double* m, d3 v) {
    d3 r = scale3(ld3(m), v.x);
    r = add3(scale3(ld3(m + 3), v.y), r);
    r = add3(scale3(ld3(m + 6), v.z), r);
    return r;
}

// 256-bit read-only global load (sm_100: LDG.E.256): one request fetches a 32-byte sector per lane, so a 128-byte
// node or plane record costs a diverged warp 4 trips through the L1 pipeline instead of 8.  p must be 32-byte aligned.
struct __align__(32) f32x8 {
    float v[8];
};
__device__ __forceinline__ f32x8 ldg256(const void* p) {
    f32x8 r;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
        : "l"(p));
    return r;
}
struct __align__(32) f64x4 {
    double v[4];
};
__device__ __forceinline__ f64x4 ldg256d(const void* p) {
    f64x4 r;
    asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
    return r;
}

// --------------------------------------------------------------------------- wrappers
// Ray into the object space of one instance (translate.rs:37-42, rotate.rs:91-97, scale.rs:73-78).
__device__ __forceinline__ void xform_ray(const nrrt_xform* x, d3& o, d3& d) {
    if (x->kind == NRRT_XF_TRANSLATE) {
        o = sub3(o, ld3(x->to_obj));
    } else if (x->kind == NRRT_XF_ROTATE) {
        o = mat3_mul(x->to_obj, o);
        d = mat3_mul(x->to_obj, d);
    } else {
        o = mat4_point(x->to_obj, o);
        d = mat4_vector(x->to_obj, d);
    }
}
__device__ __forceinline__ void instance_ray_inl(const DevScene& S, uint32_t inst, d3& o, d3& d) {
    const nrrt_instance* in = &S.instances[inst];
    uint32_t f = in->first_xform, n = in->n_xforms;
    for (uint32_t k = 0; k < n; ++k) xform_ray(&S.xforms[f + k], o, d);
}
__device__ __noinline__ void instance_ray(const DevScene& S, uint32_t inst, d3& o, d3& d) {
    instance_ray_inl(S, inst, o, d);
}
// Hit back to the parent space (translate.rs:45-48, rotate.rs:100-105, scale.rs:82-85: point only).
__device__ __noinline__ void instance_hit_back(const DevScene& S, uint32_t inst, d3& point, d3& normal) {
    const nrrt_instance* in = &S.instances[inst];
    uint32_t f = in->first_xform, n = in->n_xforms;
    for (uint32_t k = n; k-- > 0;) {
        const nrrt_xform* x = &S.xforms[f + k];
        if (x->kind == NRRT_XF_TRANSLATE) {
            point = add3(point, ld3(x->to_obj));
        } else if (x->kind == NRRT_XF_ROTATE) {
            point = mat3_mul(x->to_world, point);
            normal = mat3_mul(x->to_world, normal);
        } else {
            point = mat4_point(x->to_world, point);
        }
    }
}

// --------------------------------------------------------------------------- exact box test
// AABB::hit (aabb.rs:110-132) with Interval::ensure / intersection / is_empty (interval.rs:22-46).
__device__ __noinline__ bool box_hit_exact(const nrrt_box* b, d3 o, d3 d, double tmin, double tmax) {
    double lo = tmin, hi = tmax;
    const double oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double t0 = xdiv(xsub(b->lo[a], oo[a]), dd[a]);
        double t1 = xdiv(xsub(b->hi[a], oo[a]), dd[a]);
        double mn, mx;
        if (t0 < t1) {
            mn = t0, mx = t1;
        } else {
            mn = t1, mx = t0;
        }
        lo = fmax(lo, mn);  // f64::max: NaN-ignoring, like CUDA fmax
        hi = fmin(hi, mx);
        if (lo > hi) return false;
    }
    return true;
}

// --------------------------------------------------------------------------- primitives
// center(t) = Ray::new(center, speed.unwrap_or(ZERO)).at(time) (sphere.rs:110-111); compiled only into kernels that
// handle NRRT_F_MOTION, and a no-op for scenes without moving spheres.
template <uint32_t F>
__device__ __forceinline__ d3 sphere_center(const DevScene& S, uint32_t i, d3 c, double time) {
    if ((F & NRRT_F_MOTION) && S.sphere_speed != nullptr) c = add3(c, scale3(ld3(S.sphere_speed + 3 * (size_t)i), time));
    return c;
}

// Sphere::hit (objects/sphere.rs:105-147): returns t or NaN for a miss.
template <uint32_t F = NRRT_F_ALL>
__device__ __forceinline__ double sphere_t(const DevScene& S, uint32_t i, d3 o, d3 d, double tmin, double tmax,
                                           double time) {
    NRRT_CHECK(i < S.n_spheres, "sphere index");
    const f64x4 rec = ldg256d(S.sphere_rec + 4 * (size_t)i);
    d3 c = sphere_center<F>(S, i, mk3(rec.v[0], rec.v[1], rec.v[2]), time);
    double r = rec.v[3];
    d3 ec = sub3(c, o);
    double a = dot3(d, d);
    double h = dot3(ec, d);
    double cc = xsub(dot3(ec, ec), xmul(r, r));
    double disc = xsub(xmul(h, h), xmul(a, cc));
    if (disc < 0.0) return __longlong_as_double(0x7ff8000000000000LL);
    double sq = xsqrt(disc);
    double t = xdiv(xsub(h, sq), a);
    if (tmin < t && t < tmax) return t;  // Interval::surrounds
    t = xdiv(xadd(h, sq), a);
    if (tmin < t && t < tmax) return t;
    return __longlong_as_double(0x7ff8000000000000LL);
}

// Plane::hit (objects/plane.rs:141-174): returns t or NaN; alpha/beta and the hit point through pointers.
// `tbest` = t of the best hit so far: a candidate with t > tbest can never win (equal t still can, by leaf
// order), so its interior test is skipped — same result as the reference, fewer flops.
__device__ __forceinline__ double plane_t(const DevScene& S, uint32_t i, d3 o, d3 d, double tmin, double tmax,
                                          double tbest, double* alpha_out, double* beta_out, d3* point_out) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    NRRT_CHECK(i < S.n_planes, "plane index");
    const double* rec = S.plane_rec + 16 * (size_t)i;
    const f64x4 q0 = ldg256d(rec);  // normal xyz, d
    d3 n = mk3(q0.v[0], q0.v[1], q0.v[2]);
    double denom = dot3(n, d);
    if (fabs(denom) < 1e-8) return nan;
    double t = xdiv(xsub(q0.v[3], dot3(n, o)), denom);
    if (!(tmin <= t && t <= tmax)) return nan;  // Interval::contains
    if (t > tbest) return nan;
    const f64x4 q1 = ldg256d(rec + 4), q2 = ldg256d(rec + 8), q3 = ldg256d(rec + 12);
    d3 pp = mk3(q1.v[0], q1.v[1], q1.v[2]), w = mk3(q1.v[3], q2.v[0], q2.v[1]), uu = mk3(q2.v[2], q2.v[3], q3.v[0]),
       vv = mk3(q3.v[1], q3.v[2], q3.v[3]);
    d3 point = ray_at(o, d, t);
    d3 q = sub3(point, pp);
    double alpha = dot3(w, cross3(q, vv));
    double beta = dot3(w, cross3(uu, q));
    bool interior;
    if (S.plane_material[i] & NRRT_PLANE_TRIANGLE_BIT)
        interior = alpha > 0.0 && beta > 0.0 && xadd(alpha, beta) < 1.0;
    else
        interior = (0.0 <= alpha && alpha <= 1.0) && (0.0 <= beta && beta <= 1.0);
    if (!interior) return nan;
    *alpha_out = alpha;
    *beta_out = beta;
    *point_out = point;
    return t;
}

// --------------------------------------------------------------------------- f32 reject-only plane test
// Plane::hit (plane.rs:141-174) evaluated in f32 with a running error bound, used ONLY to prove a miss: when the bound
// shows that t lies outside [tmin, best t] or that alpha / beta lie outside the primitive, the exact f64 test would
// return None as well and is skipped; everything else ("maybe") goes to the exact test, which alone decides hits and
// produces t, alpha, beta.  Like the f32 box filter, it can only save work, never change a result.
//
// Record (4 x float4, built at upload from the f64 record): normal xyz, d | A xyz, p.x | B xyz, p.y | p.z, +-|A|_1,
// |B|_1, |p|_inf, with A = v x w and B = w x u so that alpha = q.A and beta = q.B (w.(q x v) = q.(v x w),
// w.(u x q) = q.(w x u)); the sign of the |A|_1 word carries the Triangle flag.
// Error model (u = 2^-24): inputs are f64 values rounded to f32, every bound below uses 16u per rounding step where
// first-order analysis needs at most 5u, plus an absolute 1e-6 on t (relative) and on the barycentrics, which also
// swallows the f64 rounding of the reference's own evaluation (1e-15).  NaN / inf anywhere make every comparison
// false, i.e. "maybe".
struct Ray32P {
    float ox, oy, oz, dx, dy, dz;
    float omax, dmax;  // |o|_inf, |d|_inf
};
__device__ __forceinline__ Ray32P make_ray32p(d3 o, d3 d) {
    Ray32P r;
    r.ox = (float)o.x, r.oy = (float)o.y, r.oz = (float)o.z;
    r.dx = (float)d.x, r.dy = (float)d.y, r.dz = (float)d.z;
    r.omax = fmaxf(fmaxf(fabsf(r.ox), fabsf(r.oy)), fabsf(r.oz));
    r.dmax = fmaxf(fmaxf(fabsf(r.dx), fabsf(r.dy)), fabsf(r.dz));
    return r;
}
#define NRRT_P32_U 9.5367431640625e-07f  // 16 * 2^-24
// true = the exact test is certain to return None
__device__ __forceinline__ bool plane_prereject(const DevScene& S, uint32_t i, const Ray32P& r, float tmin_lo, float tcull) {
    const float4* rec = S.plane32 + 4 * (size_t)i;
    const f32x8 a = ldg256(rec), b = ldg256(rec + 2);
    const float nx = a.v[0], ny = a.v[1], nz = a.v[2], D = a.v[3];
    const float Ax = a.v[4], Ay = a.v[5], Az = a.v[6], px = a.v[7];
    const float Bx = b.v[0], By = b.v[1], Bz = b.v[2], py = b.v[3];
    const float pz = b.v[4], a1s = b.v[5], b1 = b.v[6], pmax = b.v[7];
    const float den = fmaf(nx, r.dx, fmaf(ny, r.dy, nz * r.dz));
    const float e_den = NRRT_P32_U * 1.75f * r.dmax;  // |n|_1 <= sqrt(3): the normal is unit length
    if (!(fabsf(den) > 2.0f * e_den)) return false;
    const float num = D - fmaf(nx, r.ox, fmaf(ny, r.oy, nz * r.oz));
    const float e_num = NRRT_P32_U * (fabsf(D) + 1.75f * r.omax);
    const float rden = 1.0f / den;
    const float t = num * rden, at = fabsf(t);
    // |den_true| >= |den| - e_den >= |den| / 2
    const float e_t = 2.0f * fabsf(rden) * fmaf(at, e_den, e_num) + (NRRT_P32_U + 1e-6f) * at;
    if (t - e_t > tcull || t + e_t < tmin_lo) return true;  // t > best t (strictly), or t < tmin
    const float scale = fmaf(at, r.dmax, r.omax + pmax);
    const float e_q = fmaf(NRRT_P32_U, scale, r.dmax * e_t);
    const float qx = fmaf(t, r.dx, r.ox) - px, qy = fmaf(t, r.dy, r.oy) - py, qz = fmaf(t, r.dz, r.oz) - pz;
    const float alpha = fmaf(qx, Ax, fmaf(qy, Ay, qz * Az)), beta = fmaf(qx, Bx, fmaf(qy, By, qz * Bz));
    // each q_i is off by at most e_q, the dot product adds 3 roundings of terms bounded by scale * |A|_inf
    const float e_a = fmaf(fabsf(a1s), e_q + NRRT_P32_U * scale, 1e-6f), e_b = fmaf(b1, e_q + NRRT_P32_U * scale, 1e-6f);
    if (alpha + e_a < 0.0f || beta + e_b < 0.0f || alpha - e_a > 1.0f || beta - e_b > 1.0f) return true;
    if (__float_as_uint(a1s) >> 31) return (alpha + beta) - (e_a + e_b) > 1.0f;  // Triangle: alpha + beta < 1
    return false;
}

// --------------------------------------------------------------------------- closest hit
// Instance chain of a leaf (one id per nesting level).  Scalar members with select-based accessors instead of an
// array: an array member that is ever indexed dynamically pins the whole enclosing state struct in local memory.
static_assert(NRRT_MAX_INSTANCE_DEPTH == 4, "InstChain has four members");
struct InstChain {
    uint32_t a, b, c, d;
    __device__ __forceinline__ uint32_t get(uint32_t k) const { return k == 0 ? a : (k == 1 ? b : (k == 2 ? c : d)); }
    __device__ __forceinline__ void set(uint32_t k, uint32_t v) {
        a = k == 0 ? v : a, b = k == 1 ? v : b, c = k == 2 ? v : c, d = k == 3 ? v : d;
    }
    __device__ __forceinline__ void clear() { a = b = c = d = 0; }
};
struct HitId {
    double t;        // +inf = miss
    uint32_t prim;   // NRRT_REF_NONE = miss
    uint32_t depth;  // instance levels above prim
    InstChain inst;
};

struct TraceCounters {
    uint32_t nodes, exact, prims, inst, inst_miss;
};

__device__ __forceinline__ uint32_t leaf_order(const DevScene& S, uint32_t ref) {
    uint32_t ty = NRRT_REF_TYPE(ref), ix = NRRT_REF_INDEX(ref);
    if (ty == NRRT_REF_SPHERE) return S.sphere_order[ix];
    if (ty == NRRT_REF_PLANE) return S.plane_order[ix];
    return S.instance_order[ix];
}

// Equal-t tie: the reference keeps the right child (object.rs:110-114), i.e. the candidate that comes
// later in depth-first leaf order wins.  Compare the two leaf paths level by level.
// Both instance chains come BY VALUE: passing pointers into the traversal state would pin the whole state struct in
// local memory (the compiler cannot split an object whose interior address escapes into a call).
__device__ __noinline__ bool tie_candidate_wins(const DevScene& S, uint32_t cand, InstChain cur_chain, uint32_t level,
                                                InstChain best_chain, uint32_t best_prim, uint32_t best_depth) {
    for (uint32_t l = 0;; ++l) {
        bool ca = l < level, cb = l < best_depth;
        uint32_t ra = ca ? NRRT_REF(NRRT_REF_INSTANCE, cur_chain.get(l)) : cand;
        uint32_t rb = cb ? NRRT_REF(NRRT_REF_INSTANCE, best_chain.get(l)) : best_prim;
        if (ra != rb) return leaf_order(S, ra) > leaf_order(S, rb);
        if (!ca || !cb) return false;  // same leaf
    }
}

// Per-level f32 view of the ray for the box filter.
struct Ray32 {
    float idx, idy, idz;  // 1/d
    float ox, oy, oz;     // o/d
    float margin;         // absolute error term that depends on the ray only; +inf for a degenerate ray (a zero /
                          // denormal / overflowing direction component): then no filter comparison is ever
                          // conclusive — every child is visited, every inner box goes to the exact test, nothing is
                          // pruned — without a flag to test in the node loop
};
// relative error budget of one f32 slab distance: rounding of box and origin (2^-24 each), the approximate
// reciprocal (MUFU.RCP, <= 2^-23), the products (2^-24 each) — about 5 x 2^-24 = 3e-7 — plus slack
#define NRRT_BOX_EPS 5.0e-7f
// 1/x for the filter only: the hardware approximation (1 instruction) instead of the IEEE-rounded reciprocal (about
// ten); its error is part of NRRT_BOX_EPS.  Zero and denormal inputs give +-inf, which marks the ray degenerate.
__device__ __forceinline__ float rcp_fast(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ Ray32 make_ray32(d3 o, d3 d) {
    Ray32 r;
    r.idx = rcp_fast((float)d.x), r.idy = rcp_fast((float)d.y), r.idz = rcp_fast((float)d.z);
    r.ox = (float)o.x * r.idx, r.oy = (float)o.y * r.idy, r.oz = (float)o.z * r.idz;
    float om = fmaxf(fmaxf(fabsf(r.ox), fabsf(r.oy)), fabsf(r.oz));
    r.margin = NRRT_BOX_EPS * 2.0f * om + 1e-30f;
    float s = (r.idx + r.idy + r.idz) + (r.ox + r.oy + r.oz);  // inf or nan if any term is
    if (!(fabsf(s) < 3.0e38f) || !(om < 3.0e38f)) r.margin = __int_as_float(0x7f800000);
    return r;
}

// f32 slab filter on one child box.  Returns gap = hi_min - lo_max (>= m: certain hit, < -m: certain
// miss, otherwise inconclusive), the entry distance lo_max and the margin m.
__device__ __forceinline__ void box_filter(const Ray32& r, float lx, float ly, float lz, float hx, float hy, float hz,
                                           float tmin, float tmax, float& lo_max, float& gap, float& m) {
    float ax = fmaf(lx, r.idx, -r.ox), bx = fmaf(hx, r.idx, -r.ox);
    float ay = fmaf(ly, r.idy, -r.oy), by = fmaf(hy, r.idy, -r.oy);
    float az = fmaf(lz, r.idz, -r.oz), bz = fmaf(hz, r.idz, -r.oz);
    float lo = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), tmin));
    float hi = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), tmax));
    lo_max = lo;
    gap = hi - lo;
    m = fmaf(NRRT_BOX_EPS, fmaxf(fabsf(lo), fabsf(hi)), r.margin);
}

// Box test of a BVH *root* (scene root / nested BVH behind an instance; object.rs:102): f32 filter on the
// on-the-fly rounded box first, the reference's exact f64 slab test only when the filter is inconclusive.
template <bool COUNT>
__device__ __forceinline__ bool root_box_test(const nrrt_box* b, const Ray32& r32, d3 o, d3 d, double tmin,
                                              double tmax, float tmin32, float tmax32, TraceCounters* cnt) {
    {
        float e, g, m;
        box_filter(r32, (float)b->lo[0], (float)b->lo[1], (float)b->lo[2], (float)b->hi[0], (float)b->hi[1],
                   (float)b->hi[2], tmin32, tmax32, e, g, m);
        if (g >= m) return true;
        if (g < -m) return false;
    }
    if (COUNT) cnt->exact++;
    return box_hit_exact(b, o, d, tmin, tmax);
}

// ---- one visit of a four-slot node (nrrt_wnode, include/nrrt.h)
__device__ __forceinline__ uint32_t pick4(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t i) {
    const uint32_t lo = (i & 1u) ? b : a, hi = (i & 1u) ? d : c;
    return (i & 2u) ? hi : lo;
}
__device__ __forceinline__ void cswap(uint32_t& a, uint32_t& b) {
    const uint32_t lo = min(a, b), hi = max(a, b);
    a = lo, b = hi;
}
// Tests the four slot boxes of wide node `ni` with the f32 filter (inconclusive slots: the reference's exact f64 tests,
// gate first, then the slot's own box if it is an inner node), drops what starts certainly behind the best hit
// (tcull; not with VISIT_ALL), and returns the visited slots' refs sorted near to far in out[0..n).
// load_exact_ray(o, d) fetches the f64 ray of the current space; it is only called on the rare inconclusive path.
template <bool VISIT_ALL, bool COUNT, class LoadRay>
__device__ __forceinline__ uint32_t wide_visit(const DevScene& S, const Ray32& r32, float tmin32, float tmax32,
                                               float tcull, uint32_t ni, double tmin, double tmax, LoadRay&& load_exact_ray,
                                               TraceCounters* cnt, uint32_t (&out)[4]) {
    NRRT_CHECK(ni < S.n_wnodes, "wide node index");
    const float4* np = S.wnodes + 8 * (size_t)ni;
    const f32x8 A = ldg256(np), B = ldg256(np + 2), C = ldg256(np + 4);  // lo x,y | lo z, hi x | hi y,z
    const uint4 CH = __ldg(reinterpret_cast<const uint4*>(np + 6));
    const float lx[4] = {A.v[0], A.v[1], A.v[2], A.v[3]}, ly[4] = {A.v[4], A.v[5], A.v[6], A.v[7]};
    const float lz[4] = {B.v[0], B.v[1], B.v[2], B.v[3]}, hx[4] = {B.v[4], B.v[5], B.v[6], B.v[7]};
    const float hy[4] = {C.v[0], C.v[1], C.v[2], C.v[3]}, hz[4] = {C.v[4], C.v[5], C.v[6], C.v[7]};
    const uint32_t ch[4] = {CH.x, CH.y, CH.z, CH.w};
    if (COUNT) cnt->nodes++;
    float e[4], m[4];
    bool v[4], amb[4], any_amb = false;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        float g;
        box_filter(r32, lx[s], ly[s], lz[s], hx[s], hy[s], hz[s], tmin32, tmax32, e[s], g, m[s]);
        // leaves are not box-tested by the reference (object.rs:95-97): visit unless certainly missed; inner slots
        // and gated slots must pass the reference's tests: certain from the filter, else exact
        v[s] = (ch[s] != NRRT_REF_NONE) && !(g < -m[s]);
        amb[s] = v[s] && !(g >= m[s]);
        any_amb = any_amb || amb[s];
    }
    if (any_amb) {  // rare
        const uint4 ME = __ldg(reinterpret_cast<const uint4*>(np + 7));
        const uint32_t me[4] = {ME.x, ME.y, ME.z, ME.w};
        d3 o, d;
        load_exact_ray(o, d);
        // (a rolled loop over bit masks: one copy of the call sequence; the slot arrays stay in registers)
        uint32_t amb_mask = 0, ok_mask = 0, gate_mask = 0, node_mask = 0;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            amb_mask |= amb[s] ? 1u << s : 0u;
            gate_mask |= (me[s] & NRRT_WNODE_GATED) ? 1u << s : 0u;
            node_mask |= NRRT_REF_TYPE(ch[s]) == NRRT_REF_NODE ? 1u << s : 0u;
        }
#pragma unroll 1
        for (uint32_t s = 0; s < 4; ++s) {
            if (!((amb_mask >> s) & 1u)) continue;
            bool ok = true;
            if ((gate_mask >> s) & 1u) {
                if (COUNT) cnt->exact++;
                ok = box_hit_exact(S.wide_boxes + 8 * (size_t)ni + 2 * s + 1, o, d, tmin, tmax);
            }
            if (ok && ((node_mask >> s) & 1u)) {
                if (COUNT) cnt->exact++;
                ok = box_hit_exact(S.wide_boxes + 8 * (size_t)ni + 2 * s, o, d, tmin, tmax);
            }
            ok_mask |= ok ? 1u << s : 0u;
        }
#pragma unroll
        for (int s = 0; s < 4; ++s)
            if (amb[s]) v[s] = (ok_mask >> s) & 1u;
    }
    uint32_t k[4], n = 0;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        // prune slots that start certainly behind the best hit (ties are kept: margin > 0)
        if (!VISIT_ALL) v[s] = v[s] && !(e[s] - m[s] > tcull);
        n += v[s] ? 1u : 0u;
        // sort key: entry distance (non-negative for tmin >= 0, so its bit pattern orders like the value) with the
        // slot number in the two low bits; the order only affects how soon the best hit shrinks the search
        k[s] = v[s] ? (VISIT_ALL ? (uint32_t)s : ((__float_as_uint(e[s]) & ~3u) | (uint32_t)s)) : 0xFFFFFFFFu;
    }
    cswap(k[0], k[1]);
    cswap(k[2], k[3]);
    cswap(k[0], k[2]);
    cswap(k[1], k[3]);
    cswap(k[1], k[2]);
#pragma unroll
    for (int s = 0; s < 4; ++s) out[s] = pick4(ch[0], ch[1], ch[2], ch[3], k[s] & 3u);
    return n;
}

// Per-query context handed to begin()/round() on every call instead of being stored in the traversal state, so
// base pointers are re-read from the kernel's constant bank rather than pinned in registers.
//   get(): the world-space ray (needed again when an instance is left)
//   put(): attributes of a candidate that just became the best hit
// Fixed-ray queries / megakernel: ray in registers, attributes recomputed later by resolve_hit.
// kRayInCtx: the context also keeps the CURRENT-space ray (world at level 0, object space inside an instance), so
// the traversal state does not pin 12 registers for it across the node loop (fused kernel: shared memory).
struct RegCtx {
    static constexpr bool kRayInCtx = false;
    d3 o, d;
    double tm;  // Ray::time
    __device__ __forceinline__ double time() const { return tm; }
    __device__ __forceinline__ void get(d3& oo, d3& dd) const { oo = o, dd = d; }
    __device__ __forceinline__ void get_obj(d3&, d3&) const {}
    __device__ __forceinline__ void put_obj(d3, d3) const {}
    __device__ __forceinline__ void put(uint32_t, d3, double, double, d3) const {}
};
// Wavefront: ray re-read from the SoA path state (saves 12 registers across the node loop); attributes go straight
// into the slot's hit record so the shade kernel neither re-applies the wrapper chain to the ray nor recomputes
// alpha/beta.  attr = [8][n]: object-space hit point xyz, alpha, beta, and (hits inside an instance only) the
// object-space ray direction xyz that decides front_face.
struct MemCtx {
    static constexpr bool kRayInCtx = false;
    __device__ __forceinline__ void get_obj(d3&, d3&) const {}
    __device__ __forceinline__ void put_obj(d3, d3) const {}
    const double* ray;  // [7][n]: origin, direction, time
    double* attr;       // [8][n]
    uint32_t n, slot;
    __device__ __forceinline__ double time() const { return ray[6 * (size_t)n + slot]; }
    __device__ __forceinline__ void get(d3& oo, d3& dd) const {
        oo = mk3(ray[slot], ray[(size_t)n + slot], ray[2 * (size_t)n + slot]);
        dd = mk3(ray[3 * (size_t)n + slot], ray[4 * (size_t)n + slot], ray[5 * (size_t)n + slot]);
    }
    __device__ __forceinline__ void put(uint32_t level, d3 p, double a, double b, d3 dobj) const {
#if NRRT_HIT_SINK
        attr[slot] = p.x, attr[(size_t)n + slot] = p.y, attr[2 * (size_t)n + slot] = p.z;
        attr[3 * (size_t)n + slot] = a, attr[4 * (size_t)n + slot] = b;
        if (level) attr[5 * (size_t)n + slot] = dobj.x, attr[6 * (size_t)n + slot] = dobj.y, attr[7 * (size_t)n + slot] = dobj.z;
#endif
    }
};

// BVH::hit (objects/object.rs:89-121) over the flattened scene, as a resumable state machine.
//   VISIT_ALL = true : visits exactly the reference's node set (no pruning by the best hit so far)
//   VISIT_ALL = false: near-first order + conservative pruning by the best t (same result, fewer visits)
//
// begin() starts a query; round() advances it by one "round": the inner loop walks inner nodes only — cheap f32
// work every lane of a warp does in lock step — until the lane holds a leaf; then the warp VOTES which kind of
// leaf to process this round (exact f64 primitive tests, or instance entries) and only the lanes holding that
// kind advance, the others keep their leaf for a later round.  The two expensive, mutually divergent code paths
// therefore never serialise inside one round, and each runs with as many lanes as possible.
// round() must be called by ALL 32 lanes of the warp (lanes without a query pass has = false); it returns true
// when the lane's query is finished.  Keeping the state resumable lets a persistent warp swap finished rays for
// fresh ones between rounds.
//   SPEC: speculative traversal: a lane that reaches a primitive leaf parks it and keeps walking inner nodes while
//         other lanes of its warp are still in the node loop, instead of idling.  Pays on deep trees (teapot +16 %,
//         sphere field +7 %), costs on tiny ones (Cornell, 17 nodes: -4 %), so the render path selects it by tree size.
//   WIDE: walk the four-slot nodes (default) or the binary ones (small trees; needs DevScene::bnodes)
template <bool VISIT_ALL, bool COUNT, uint32_t F = NRRT_F_ALL, bool SPEC = false, bool WIDE = true>
struct Traversal {
    d3 o, d;         // ray in the current space (world, or the object space of the innermost entered instance)
    Ray32 r32;
    float tcull;
    uint32_t sp, cur, level;
    uint32_t pend;   // NRRT_SPECULATE: a postponed primitive leaf of the current level, or NRRT_REF_NONE
    InstChain cur_inst;
    HitId best;
    static constexpr bool kSpeculate = SPEC && !VISIT_ALL;
    static __device__ __forceinline__ bool is_prim_ref(uint32_t ref) {
        const uint32_t ty = NRRT_REF_TYPE(ref);
        return ((F & NRRT_F_SPHERES) && ty == NRRT_REF_SPHERE) || ((F & NRRT_F_PLANES) && ty == NRRT_REF_PLANE);
    }
    // Speculative traversal: park the primitive leaf in hand and take the next stack entry, so the lane can go on
    // walking inner nodes.  The parked leaf is tested in phase 2 of the same round, before anything that changes
    // the coordinate space, so it always belongs to the current level.  Testing it later only delays pruning.
    __device__ __forceinline__ void postpone_leaf(bool has, uint32_t* stack, uint32_t sstride) {
        if (kSpeculate && has && pend == NRRT_REF_NONE && is_prim_ref(cur)) {
            pend = cur;
            cur = NRRT_REF_NONE;
            if (sp) {
                --sp;
                cur = stack[sp * sstride];
            }
        }
    }

    // the ray in the current space: from the traversal state, or from the context when it owns it
    template <class Ctx>
    __device__ __forceinline__ void load_ray(const Ctx& ctx, d3& oo, d3& dd) const {
        if (Ctx::kRayInCtx) {
            if (!(F & NRRT_F_INSTANCES) || level == 0) ctx.get(oo, dd);
            else ctx.get_obj(oo, dd);
        } else {
            oo = o, dd = d;
        }
    }
    template <class Ctx>
    __device__ __forceinline__ void store_ray(const Ctx& ctx, d3 oo, d3 dd) {  // call AFTER `level` is updated
        if (Ctx::kRayInCtx) {
            if ((F & NRRT_F_INSTANCES) && level > 0) ctx.put_obj(oo, dd);
        } else {
            o = oo, d = dd;
        }
    }

    // one visit of a binary node (nrrt_node): both children's boxes, near child first
    template <class Ctx>
    __device__ __forceinline__ void binary_step(const DevScene& S, const Ctx& ctx, double tmin, double tmax, float tmin32,
                                                float tmax32, uint32_t* stack, uint32_t sstride, TraceCounters* cnt) {
        const uint32_t ni = NRRT_REF_INDEX(cur);
        const float4* np = S.bnodes + 4 * (size_t)ni;
        const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3);
        // layout: lo[0].xyz lo[1].xyz | hi[0].xyz hi[1].xyz | child[0] child[1] pad pad
        const uint32_t c0 = __float_as_uint(n3.x), c1 = __float_as_uint(n3.y);
        if (COUNT) cnt->nodes++;
        float e0, g0, m0, e1, g1, m1;
        box_filter(r32, n0.x, n0.y, n0.z, n1.z, n1.w, n2.x, tmin32, tmax32, e0, g0, m0);
        box_filter(r32, n0.w, n1.x, n1.y, n2.y, n2.z, n2.w, tmin32, tmax32, e1, g1, m1);
        // leaves are not box-tested by the reference (object.rs:95-97): visit unless certainly missed;
        // inner children must pass the reference's test: certain from the filter, else exact
        bool v0 = (c0 != NRRT_REF_NONE) && !(g0 < -m0);
        bool v1 = (c1 != NRRT_REF_NONE) && !(g1 < -m1);
        const bool amb0 = v0 && NRRT_REF_TYPE(c0) == NRRT_REF_NODE && !(g0 >= m0);
        const bool amb1 = v1 && NRRT_REF_TYPE(c1) == NRRT_REF_NODE && !(g1 >= m1);
        if (amb0 || amb1) {  // rare
            d3 o, d;
            load_ray(ctx, o, d);
            if (amb0) {
                if (COUNT) cnt->exact++;
                v0 = box_hit_exact(S.bchild_boxes + 2 * (size_t)ni, o, d, tmin, tmax);
            }
            if (amb1) {
                if (COUNT) cnt->exact++;
                v1 = box_hit_exact(S.bchild_boxes + 2 * (size_t)ni + 1, o, d, tmin, tmax);
            }
        }
        if (!VISIT_ALL) {
            // prune children that start certainly behind the best hit (ties are kept: margin > 0)
            v0 = v0 && !(e0 - m0 > tcull);
            v1 = v1 && !(e1 - m1 > tcull);
        }
        if (v0 && v1) {
            const bool swap = !VISIT_ALL && (e1 < e0);
            stack[sp * sstride] = swap ? c0 : c1;
            ++sp;
            cur = swap ? c1 : c0;
        } else if (v0 || v1) {
            cur = v0 ? c0 : c1;
        } else {
            cur = NRRT_REF_NONE;
            if (sp) {
                --sp;
                cur = stack[sp * sstride];
            }
        }
    }

    // filter bounds of the query range; the margins cover the rounding
    static __device__ __forceinline__ float lo32(double tmin) { return (float)tmin; }
    static __device__ __forceinline__ float hi32(double tmax) { return (tmax < 3.0e38) ? (float)tmax : 3.4e38f; }

    template <class Ctx>
    __device__ __forceinline__ void begin(const DevScene& S, const Ctx& ctx, double tmin, double tmax,
                                          TraceCounters* cnt) {
        const float tmin32 = lo32(tmin), tmax32 = hi32(tmax);
        best.t = NRRT_INF;
        best.prim = NRRT_REF_NONE;
        best.depth = 0;
        best.inst.clear();
        cur_inst.clear();
        level = 0;
        d3 wo, wd;
        ctx.get(wo, wd);
        store_ray(ctx, wo, wd);
        r32 = make_ray32(wo, wd);
        tcull = 3.4e38f;                                    // f32 upper bound of best.t (+ slack)
        sp = 0;
        pend = NRRT_REF_NONE;
        cur = WIDE ? S.root : S.broot;
        // root of the scene: an inner node tests its own box (object.rs:102)
        if (NRRT_REF_TYPE(cur) == NRRT_REF_NODE) {
            if (!root_box_test<COUNT>(&S.root_box, r32, wo, wd, tmin, tmax, tmin32, tmax32, cnt)) cur = NRRT_REF_NONE;
        } else if (cur != NRRT_REF_NONE) {
            // a scene that is one leaf (e.g. a single wrapped mesh): the reference tests no box here (object.rs:95-97),
            // so only what the f32 filter PROVES missed is culled — exactly as for a leaf child of an inner node
            float e, g, m;
            box_filter(r32, (float)S.root_box.lo[0], (float)S.root_box.lo[1], (float)S.root_box.lo[2],
                       (float)S.root_box.hi[0], (float)S.root_box.hi[1], (float)S.root_box.hi[2], tmin32, tmax32, e, g, m);
            if (g < -m) cur = NRRT_REF_NONE;
        }
    }

    // `stack` is this thread's slice of shared memory, stride `sstride` (bank-conflict free).
    template <class Ctx>
    __device__ __forceinline__ bool round(const DevScene& S, const Ctx& ctx, double tmin, double tmax, uint32_t* stack,
                                          uint32_t sstride, TraceCounters* cnt, bool has) {
        const float tmin32 = lo32(tmin), tmax32 = hi32(tmax);
        // ---------------- phase 1: inner nodes
        postpone_leaf(has, stack, sstride);
        for (;;) {
            const bool at_node = has && NRRT_REF_TYPE(cur) == NRRT_REF_NODE;
            if (kSpeculate) {
                // the loop runs as long as some lane WITHOUT a parked leaf has a node; lanes with a parked leaf
                // ride along (work they do here would otherwise be idle issue slots) but never prolong it
                if (!__any_sync(0xffffffffu, at_node && pend == NRRT_REF_NONE)) break;
            }
            if (!at_node) {
                if (kSpeculate) continue;
                break;
            }
            if (!WIDE) {
                binary_step(S, ctx, tmin, tmax, tmin32, tmax32, stack, sstride, cnt);
                postpone_leaf(has, stack, sstride);
                continue;
            }
            uint32_t nxt[4];
            const uint32_t n = wide_visit<VISIT_ALL, COUNT>(
                S, r32, tmin32, tmax32, tcull, NRRT_REF_INDEX(cur), tmin, tmax,
                [&](d3& oo, d3& dd) { load_ray(ctx, oo, dd); }, cnt, nxt);
            // continue with the nearest slot, the others wait on the stack (farthest at the bottom)
            NRRT_CHECK(sp + (n ? n - 1 : 0) <= NRRT_STACK_CAP, "traversal stack overflow");
            if (n > 3) stack[sp * sstride] = nxt[3], ++sp;
            if (n > 2) stack[sp * sstride] = nxt[2], ++sp;
            if (n > 1) stack[sp * sstride] = nxt[1], ++sp;
            cur = nxt[0];
            if (n == 0) {
                cur = NRRT_REF_NONE;
                if (sp) {
                    --sp;
                    cur = stack[sp * sstride];
                }
            }
            postpone_leaf(has, stack, sstride);
        }
        // ---------------- phase 2: the warp votes for one kind of leaf
        const bool parked = kSpeculate && has && pend != NRRT_REF_NONE;
        const bool cur_prim = has && is_prim_ref(cur);
        const bool is_prim = parked || cur_prim;
        const bool is_inst = (F & NRRT_F_INSTANCES) && has && !parked && NRRT_REF_TYPE(cur) == NRRT_REF_INSTANCE;
        bool serve_inst = false;
        if (F & NRRT_F_INSTANCES) {  // scenes without wrappers have nothing to vote on
#if NRRT_LEAF_VOTE
            const unsigned m_prim = __ballot_sync(0xffffffffu, is_prim), m_inst = __ballot_sync(0xffffffffu, is_inst);
            serve_inst = __popc(m_inst) > __popc(m_prim);
#else
            serve_inst = is_inst;  // no vote: every lane processes whatever leaf it holds
#endif
        }
        if (!has) return true;
        d3 o, d;
        if (is_prim || is_inst) load_ray(ctx, o, d);
        if (is_prim) {
            if (serve_inst) return false;  // wait: this round enters instances
            // one or two leaves: the parked one first, then the one in hand (one code site, at most two trips)
            uint32_t leaf = parked ? pend : cur;
            bool again = parked && cur_prim;
            for (;;) {
                if (COUNT) cnt->prims++;
                double a_ = 0.0, b_ = 0.0;
                d3 pt;
                double t;
                if ((F & NRRT_F_SPHERES) && (!(F & NRRT_F_PLANES) || NRRT_REF_TYPE(leaf) == NRRT_REF_SPHERE)) {
                    t = sphere_t<F>(S, NRRT_REF_INDEX(leaf), o, d, tmin, tmax, (F & NRRT_F_MOTION) ? ctx.time() : 0.0);
                    pt = ray_at(o, d, t);
                } else {
                    t = plane_t(S, NRRT_REF_INDEX(leaf), o, d, tmin, tmax, VISIT_ALL ? NRRT_INF : best.t, &a_, &b_, &pt);
                }
                if (t == t) {
                    bool take = t < best.t;
                    if (!take && t == best.t)
                        take = tie_candidate_wins(S, leaf, cur_inst, level, best.inst, best.prim, best.depth);
                    if (take) {
                        best.t = t;
                        best.prim = leaf;
                        best.depth = level;
                        if ((F & NRRT_F_INSTANCES) && level) best.inst = cur_inst;
                        ctx.put(level, pt, a_, b_, d);
                        // f32 upper bound of t with slack far above any f64 rounding discrepancy
                        float tf = (float)t;
                        tcull = tf + fabsf(tf) * 1.0e-6f + 1e-30f;
                    }
                }
                if (!kSpeculate || !again) break;
                again = false;
                leaf = cur;
            }
            if (kSpeculate) {
                pend = NRRT_REF_NONE;
                if (!cur_prim) {  // the entry in hand (node / instance / level marker / nothing) is still to be served
                    if (cur == NRRT_REF_NONE) return true;
                    if (!((F & NRRT_F_INSTANCES) && cur == NRRT_REF_POP)) return false;
                }
            }
        } else if (is_inst) {
            if (!serve_inst) return false;  // wait: this round tests primitives
            // enter an instance: transform the ray (exactly, wrapper by wrapper), test the nested root's box
            uint32_t ii = NRRT_REF_INDEX(cur);
            const nrrt_instance* in = &S.instances[ii];
            uint32_t inner = WIDE ? in->inner : S.inst_binner[ii];
            if (inner != NRRT_REF_NONE && level < NRRT_MAX_INSTANCE_DEPTH) {
                d3 no = o, nd = d;
                if (COUNT) cnt->inst++;
                instance_ray_inl(S, ii, no, nd);
                Ray32 n32 = make_ray32(no, nd);
                bool enter = true;
                if (NRRT_REF_TYPE(inner) == NRRT_REF_NODE)
                    enter = root_box_test<COUNT>(&in->inner_box, n32, no, nd, tmin, tmax, tmin32, tmax32, cnt);
                if (enter) {
                    NRRT_CHECK(sp < NRRT_STACK_CAP, "traversal stack overflow (level marker)");
                    stack[sp * sstride] = NRRT_REF_POP;
                    ++sp;
                    cur_inst.set(level, ii);
                    ++level;
                    store_ray(ctx, no, nd);
                    r32 = n32;
                    cur = inner;
                    return false;
                }
                if (COUNT) cnt->inst_miss++;
            }
        }
        // next pending entry; level markers are consumed on the way (leaving an instance rebuilds the parent-level
        // ray from the world ray: a bit-identical recomputation).  Phase 1 may already have popped a marker.
        bool in_hand = (F & NRRT_F_INSTANCES) && (cur == NRRT_REF_POP);
        for (;;) {
            if (!in_hand) {
                if (sp == 0) {
                    cur = NRRT_REF_NONE;
                    return true;
                }
                --sp;
                cur = stack[sp * sstride];
            }
            in_hand = false;
            if (!(F & NRRT_F_INSTANCES) || cur != NRRT_REF_POP) return false;
            --level;
            d3 po, pd;
            ctx.get(po, pd);
#pragma unroll
            for (int l = 0; l < NRRT_MAX_INSTANCE_DEPTH; ++l)
                if (l < (int)level) instance_ray(S, cur_inst.get(l), po, pd);
            store_ray(ctx, po, pd);
            r32 = make_ray32(po, pd);
        }
    }
};

// Convenience: run one query per lane to completion (fixed-ray queries, megakernel).  Must be called by all 32
// lanes of the warp; lanes with active = false only take part in the votes.
template <bool VISIT_ALL, bool COUNT>
__device__ __forceinline__ void trace_closest(const DevScene& S, d3 wo, d3 wd, double time, double tmin, double tmax,
                                              uint32_t* stack, uint32_t sstride, HitId& best, TraceCounters* cnt,
                                              bool active) {
    Traversal<VISIT_ALL, COUNT> tr;
    const RegCtx ctx{wo, wd, time};
    if (active) tr.begin(S, ctx, tmin, tmax, cnt);
    bool running = active;
    while (__any_sync(0xffffffffu, running)) {
        if (tr.round(S, ctx, tmin, tmax, stack, sstride, cnt, running)) running = false;
    }
    best = tr.best;
}

// --------------------------------------------------------------------------- hit record
struct HitRec {
    d3 point, normal;
    double u, v;
    uint32_t material;
    bool front_face;
};

// Rebuilds HitRecord (hitable.rs:38-59) of the winning primitive: object-space point/normal/uv from the
// object-space ray, then back out through the wrappers.  want_uv=false skips the sphere's acos/atan2.
__device__ __forceinline__ void resolve_hit(const DevScene& S, const HitId& h, d3 wo, d3 wd, double time, bool want_uv,
                                            HitRec& rec) {
    d3 o = wo, d = wd;
#pragma unroll
    for (int l = 0; l < NRRT_MAX_INSTANCE_DEPTH; ++l)
        if (l < (int)h.depth) instance_ray(S, h.inst.get(l), o, d);
    uint32_t ty = NRRT_REF_TYPE(h.prim), ix = NRRT_REF_INDEX(h.prim);
    d3 point = ray_at(o, d, h.t), outward;
    double u = 0.0, v = 0.0;
    if (ty == NRRT_REF_SPHERE) {
        d3 c = sphere_center<NRRT_F_ALL>(S, ix, ld3(S.sphere_rec + 4 * (size_t)ix), time);
        outward = normalize3(sub3(point, c));  // sphere.rs:151
        if (want_uv) {                         // sphere.rs:153-159
            const double PI = 3.14159265358979323846264338327950288;
            double theta = acos(-outward.y);
            double phi = xadd(atan2(-outward.z, outward.x), PI);
            u = xdiv(phi, xmul(2.0, PI));
            v = xdiv(theta, PI);
        }
        rec.material = S.sphere_material[ix];
    } else {
        const double* pr = S.plane_rec + 16 * (size_t)ix;
        outward = ld3(pr);
        d3 q = sub3(point, ld3(pr + 4));
        d3 w = ld3(pr + 7);
        u = dot3(w, cross3(q, ld3(pr + 13)));  // alpha
        v = dot3(w, cross3(ld3(pr + 10), q));  // beta
        rec.material = S.plane_material[ix] & ~NRRT_PLANE_TRIANGLE_BIT;
    }
    double sign = signum(dot3(d, outward));
    rec.front_face = sign < 0.0;
    d3 normal = scale3(outward, -sign);
#pragma unroll
    for (int l = NRRT_MAX_INSTANCE_DEPTH - 1; l >= 0; --l)
        if (l < (int)h.depth) instance_hit_back(S, h.inst.get(l), point, normal);
    rec.point = point;
    rec.normal = normal;
    rec.u = u;
    rec.v = v;
}

// Same HitRecord, from the attributes the wavefront traverse kernel stored when the candidate won (MemHitSink):
// p_obj / alpha / beta are the very values the primitive test computed, d_dir is the ray direction in the
// primitive's space (the world direction for depth 0).
template <uint32_t F = NRRT_F_ALL>
__device__ __forceinline__ void resolve_hit_attr(const DevScene& S, const HitId& h, d3 p_obj, double alpha, double beta,
                                                 d3 d_dir, double time, bool want_uv, HitRec& rec) {
    uint32_t ty = NRRT_REF_TYPE(h.prim), ix = NRRT_REF_INDEX(h.prim);
    d3 point = p_obj, outward;
    double u = alpha, v = beta;
    if ((F & NRRT_F_SPHERES) && (!(F & NRRT_F_PLANES) || ty == NRRT_REF_SPHERE)) {
        d3 c = sphere_center<F>(S, ix, ld3(S.sphere_rec + 4 * (size_t)ix), time);
        outward = normalize3(sub3(point, c));  // sphere.rs:151
        u = 0.0, v = 0.0;
        if ((F & NRRT_F_TEXTURED) && want_uv) {  // sphere.rs:153-159
            const double PI = 3.14159265358979323846264338327950288;
            double theta = acos(-outward.y);
            double phi = xadd(atan2(-outward.z, outward.x), PI);
            u = xdiv(phi, xmul(2.0, PI));
            v = xdiv(theta, PI);
        }
        rec.material = S.sphere_material[ix];
    } else {
        outward = ld3(S.plane_rec + 16 * (size_t)ix);
        rec.material = S.plane_material[ix] & ~NRRT_PLANE_TRIANGLE_BIT;
    }
    double sign = signum(dot3(d_dir, outward));
    rec.front_face = sign < 0.0;
    d3 normal = scale3(outward, -sign);
    if (F & NRRT_F_INSTANCES)
    {
#pragma unroll
        for (int l = NRRT_MAX_INSTANCE_DEPTH - 1; l >= 0; --l)
            if (l < (int)h.depth) instance_hit_back(S, h.inst.get(l), point, normal);
    }
    rec.point = point;
    rec.normal = normal;
    rec.u = u;
    rec.v = v;
}

// --------------------------------------------------------------------------- Philox4x32-10
#ifndef NRRT_PHILOX_INLINE
#define NRRT_PHILOX_INLINE __forceinline__
#endif
#ifndef NRRT_DISK_INLINE
#define NRRT_DISK_INLINE __forceinline__
#endif
__device__ NRRT_PHILOX_INLINE uint4 philox4x32_10(uint2 key, uint4 c) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ key.x, lo1, hi0 ^ c.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return c;
}
// counter = (pixel, sample, stage<<12 | iter, 0): stage 0 = camera, stage k+1 = scatter at bounce k
struct Sampler {
    uint2 key;
    uint32_t pixel, sample;
    __device__ __forceinline__ uint4 draw(uint32_t stage, uint32_t iter) const {
        return philox4x32_10(key, make_uint4(pixel, sample, (stage << 12) | (iter & 0xFFFu), 0u));
    }
};
__device__ __forceinline__ double u_m1_1(uint32_t r) { return xsub(xmul((double)r, 1.0 / 2147483648.0), 1.0); }
__device__ __forceinline__ double u_mh_h(uint32_t r) { return xsub(xmul((double)r, 1.0 / 4294967296.0), 0.5); }
__device__ __forceinline__ double u_0_1(uint32_t r) { return xmul((double)r, 1.0 / 4294967296.0); }

// vector.rs:61-70 — p/|p|^2, |p|^2 in (1e-160, 1]
__device__ __forceinline__ d3 random_in_unit_sphere(const Sampler& s, uint32_t stage) {
    for (uint32_t it = 0;; ++it) {
        uint4 r = s.draw(stage, it);
        d3 p = mk3(u_m1_1(r.x), u_m1_1(r.y), u_m1_1(r.z));
        double l2 = dot3(p, p);
        if ((1e-160 < l2 && l2 <= 1.0) || it == 0xFFFu) return div3(p, l2);
    }
}
// vector.rs:72-81 — p/|p|^2, |p|^2 < 1
__device__ NRRT_DISK_INLINE d3 random_in_unit_disk(const Sampler& s) {
    for (uint32_t it = 1;; ++it) {
        uint4 r = s.draw(0, it);
        d3 p = mk3(u_m1_1(r.x), u_m1_1(r.y), 0.0);
        double l2 = dot3(p, p);
        if (l2 < 1.0 || it == 0xFFFu) return div3(p, l2);
    }
}

// --------------------------------------------------------------------------- textures
// noise 0.9.0 Perlin (restated from the published algorithm; see DESIGN.md).
// Gradient dot product, branch-free (the hash differs per lane: a 12-way switch would serialise the warp eight
// times per octave).  h & 15: 0-3 = (+-x) +- y, 4-7 = (+-x) +- z, 8-11 = (+-y) +- z, 12-15 repeat 0, 1, 9, 11; bit 0
// negates the first term, bit 1 subtracts the second.  Every result is one exact IEEE add or subtract of the same
// operands as the table form, so the value is bit-identical.
__device__ __forceinline__ double grad3(uint32_t h, double x, double y, double z) {
    h &= 15u;
    const uint32_t k = h < 12u ? h : ((0xB910u >> ((h - 12u) * 4u)) & 15u);  // 12 -> 0, 13 -> 1, 14 -> 9, 15 -> 11
    const uint32_t g = k >> 2;
    const double a = g == 2u ? y : x;
    const double b = g == 0u ? y : z;
    const double sa = (k & 1u) ? -a : a;
    return (k & 2u) ? xsub(sa, b) : xadd(sa, b);
}
__device__ __forceinline__ double quintic(double t) {
    return xmul(xmul(xmul(t, t), t), xadd(xmul(t, xsub(xmul(t, 6.0), 15.0)), 10.0));
}
__device__ __noinline__ double perlin3(const uint8_t* __restrict__ pm, double px, double py, double pz) {
    double fx = floor(px), fy = floor(py), fz = floor(pz);
    long long cx = (long long)fx, cy = (long long)fy, cz = (long long)fz;
    double dx = xsub(px, fx), dy = xsub(py, fy), dz = xsub(pz, fz);
    double g[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        int ox = k & 1, oy = (k >> 1) & 1, oz = (k >> 2) & 1;
        uint32_t i = (uint32_t)((cx + ox) & 0xff);
        i = (uint32_t)__ldg(pm + i) ^ (uint32_t)((cy + oy) & 0xff);
        i = (uint32_t)__ldg(pm + i) ^ (uint32_t)((cz + oz) & 0xff);
        uint32_t h = __ldg(pm + i);
        g[k] = grad3(h, xsub(dx, (double)ox), xsub(dy, (double)oy), xsub(dz, (double)oz));
    }
    // g index: bit0 = x, bit1 = y, bit2 = z
    double g000 = g[0], g100 = g[1], g010 = g[2], g110 = g[3], g001 = g[4], g101 = g[5], g011 = g[6], g111 = g[7];
    double u = quintic(dx), v = quintic(dy), w = quintic(dz);
    double k0 = g000;
    double k1 = xsub(g100, g000);
    double k2 = xsub(g010, g000);
    double k3 = xsub(g001, g000);
    double k4 = xsub(xsub(xadd(g000, g110), g100), g010);
    double k5 = xsub(xsub(xadd(g000, g101), g100), g001);
    double k6 = xsub(xsub(xadd(g000, g011), g010), g001);
    double k7 = xsub(xsub(xsub(xsub(xadd(xadd(xadd(g100, g010), g001), g111), g000), g110), g101), g011);
    double r = k0;
    r = xadd(r, xmul(k1, u));
    r = xadd(r, xmul(k2, v));
    r = xadd(r, xmul(k3, w));
    r = xadd(r, xmul(xmul(k4, u), v));
    r = xadd(r, xmul(xmul(k5, u), w));
    r = xadd(r, xmul(xmul(k6, v), w));
    r = xadd(r, xmul(xmul(xmul(k7, u), v), w));
    r = xmul(r, 1.1547005383792515);
    return r < -1.0 ? -1.0 : (r > 1.0 ? 1.0 : r);
}
// Fbm<Perlin>::get
__device__ __noinline__ double fbm3(const DevScene& S, uint32_t tex, uint32_t octaves, double freq, double lac,
                                    double pers, double scale_factor, d3 p) {
    const uint8_t* tables = S.perm + 256 * (size_t)S.perm_base[tex];
    double x = xmul(p.x, freq), y = xmul(p.y, freq), z = xmul(p.z, freq);
    double result = 0.0, att = pers;
    for (uint32_t i = 0; i < octaves; ++i) {
        double s = perlin3(tables + 256 * (size_t)i, x, y, z);
        s = xmul(s, att);
        att = xmul(att, pers);
        result = xadd(result, s);
        x = xmul(x, lac), y = xmul(y, lac), z = xmul(z, lac);
    }
    return xmul(result, scale_factor);
}

__device__ __forceinline__ unsigned long long sat_u64(double x) {  // Rust `as u64`
    if (!(x == x) || x <= 0.0) return 0ull;
    if (x >= 18446744073709551615.0) return 0xFFFFFFFFFFFFFFFFull;
    return (unsigned long long)x;
}
__device__ __forceinline__ uint32_t sat_u32(double x) {  // Rust `as u32`
    if (!(x == x) || x <= 0.0) return 0u;
    if (x >= 4294967295.0) return 0xFFFFFFFFu;
    return (uint32_t)x;
}

// Texture::get_color (textures/*.rs).  Checker recursion is a loop: sub-textures always precede.
template <uint32_t F = NRRT_F_ALL>
__device__ __forceinline__ d3 texture_color(const DevScene& S, uint32_t tex, double u, double v, d3 point) {
    if (!(F & NRRT_F_TEXTURED)) return ld3(S.textures[tex].color);  // every texture of the scene is a SolidColor
    for (int guard = 0; guard < 64; ++guard) {
        const nrrt_texture* t = &S.textures[tex];
        uint32_t kind = t->kind;
        if (kind == NRRT_TEX_SOLID) return ld3(t->color);
        if (kind == NRRT_TEX_CHECKER) {  // checker.rs:77-89
            unsigned long long s = sat_u64(xmul(u, t->f0)) + sat_u64(xmul(v, t->f0));
            tex = (s % 2ull == 0ull) ? t->a : t->b;
            continue;
        }
        if (kind == NRRT_TEX_IMAGE) {  // image.rs:30-40 — nearest texel, u8/255 as f32, no sRGB decode
            uint2 sz = S.image_size[t->a];
            double cu = u < 0.0 ? 0.0 : (u > 1.0 ? 1.0 : u);
            double cv = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
            uint32_t x = sat_u32(xmul(cu, (double)sz.x));
            uint32_t y = sat_u32(xmul(xsub(1.0, cv), (double)sz.y));
            if (x >= sz.x) x = sz.x - 1;  // the reference panics here (u == 1 / v == 0)
            if (y >= sz.y) y = sz.y - 1;
            uchar4 px = tex2D<uchar4>(S.image_tex[t->a], (float)x + 0.5f, (float)y + 0.5f);
            return mk3((double)__fdiv_rn((float)px.x, 255.0f), (double)__fdiv_rn((float)px.y, 255.0f),
                       (double)__fdiv_rn((float)px.z, 255.0f));
        }
        // NOISE (noise.rs:135-145) / MARBLE (marble.rs:86-97); f1/f2 hold lacunarity/persistence,
        // color[0] holds the precomputed Fbm scale factor (filled at upload)
        double n = fabs(fbm3(S, tex, t->octaves, t->f0, t->f1, t->f2, t->color[0], point));
        if (kind == NRRT_TEX_NOISE) return mk3(n, n, n);
        double val = xdiv(xadd(1.0, sin(xadd(xmul(t->f0, point.z), xmul(10.0, n)))), 2.0);
        return mk3(val, val, val);
    }
    return mk3(0.0, 0.0, 0.0);
}

// --------------------------------------------------------------------------- materials
// Returns true if the path continues.  emitted is always set (material.rs:20-26, diffuse_light.rs:63-75).
template <uint32_t F = NRRT_F_ALL>
__device__ __forceinline__ bool shade_hit(const DevScene& S, const HitRec& h, d3 rd, bool primary, const Sampler& smp,
                                          uint32_t stage, d3& emitted, d3& atten, d3& new_dir) {
    NRRT_CHECK(h.material < S.n_materials, "material index");
    const nrrt_material* m = &S.materials[h.material];
    uint32_t kind = m->kind;
    emitted = mk3(0.0, 0.0, 0.0);
    // Lambertian and Metal both draw random_in_unit_sphere as their only random input (lambertian.rs:46,
    // metal.rs:80-81) with the same counter, so the divergent rejection loop runs once for both kinds.
    d3 rnd = mk3(0.0, 0.0, 0.0);
    if (kind == NRRT_MAT_LAMBERTIAN || kind == NRRT_MAT_METAL) rnd = random_in_unit_sphere(smp, stage);
    if (kind == NRRT_MAT_LAMBERTIAN) {  // lambertian.rs:39-55
        d3 dir = add3(h.normal, rnd);
        if (fabs(dir.x) < 1e-8 && fabs(dir.y) < 1e-8 && fabs(dir.z) < 1e-8) dir = h.normal;
        new_dir = dir;
        atten = texture_color<F>(S, m->texture, h.u, h.v, h.point);
        return true;
    }
    if (kind == NRRT_MAT_METAL) {  // metal.rs:73-91
        d3 refl = sub3(rd, scale3(h.normal, xmul(2.0, dot3(rd, h.normal))));  // glam reflect
        d3 dir = add3(normalize3(refl), scale3(rnd, m->param));
        if (dot3(dir, h.normal) > 0.0) {
            new_dir = dir;
            atten = texture_color<F>(S, m->texture, h.u, h.v, h.point);
            return true;
        }
        return false;
    }
    if ((F & NRRT_F_DIELECTRIC) && kind == NRRT_MAT_DIELECTRIC) {  // dielectric.rs:39-67
        double ri = h.front_face ? xdiv(1.0, m->param) : m->param;
        d3 unit = normalize3(rd);
        double cos_theta = fmin(dot3(neg3(unit), h.normal), 1.0);
        double sin_theta = xsqrt(xsub(1.0, xmul(cos_theta, cos_theta)));
        bool refl = xmul(ri, sin_theta) > 1.0;
        if (!refl) {
            double r0 = xdiv(xsub(1.0, ri), xadd(1.0, ri));  // reflectance :13-19
            r0 = xmul(r0, r0);
            double x = xsub(1.0, cos_theta);
            double x2 = xmul(x, x);
            double x5 = xmul(x, xmul(x2, x2));
            double p = xadd(r0, xmul(xsub(1.0, r0), x5));
            refl = p > u_0_1(smp.draw(stage, 0).x);
        }
        if (refl) {
            new_dir = sub3(unit, scale3(h.normal, xmul(2.0, dot3(unit, h.normal))));
        } else {  // glam refract
            double ndi = dot3(h.normal, unit);
            double k = xsub(1.0, xmul(xmul(ri, ri), xsub(1.0, xmul(ndi, ndi))));
            if (k >= 0.0)
                new_dir = sub3(scale3(unit, ri), scale3(h.normal, xadd(xmul(ri, ndi), xsqrt(k))));
            else
                new_dir = mk3(0.0, 0.0, 0.0);
        }
        atten = mk3(1.0, 1.0, 1.0);
        return true;
    }
    // DiffuseLight: emits, never scatters.  Seen by a camera ray it shows at x1 (quirk Q3).
    double k = primary ? 1.0 : m->param;
    emitted = scale3(texture_color<F>(S, m->texture, h.u, h.v, h.point), k);
    return false;
}

// --------------------------------------------------------------------------- camera
// Camera::get_ray (camera.rs:244-267)
// MOTION: also return Ray::time = random_range(0.0..1.0) (:264) — the third word of the jitter draw.
template <bool MOTION>
__device__ __forceinline__ void camera_ray(const nrrt_camera& cam, uint32_t x, uint32_t y, const Sampler& s, d3& o,
                                           d3& d, double& time) {
    double ox = 0.0, oy = 0.0;
    time = 0.0;
    if (MOTION || cam.samples_per_pixel > 1) {
        uint4 r = s.draw(0, 0);
        if (cam.samples_per_pixel > 1) {
            ox = u_mh_h(r.x);
            oy = u_mh_h(r.y);
        }
        if (MOTION) time = u_0_1(r.z);
    }
    d3 point = add3(add3(ld3(cam.viewport_top_left), scale3(ld3(cam.pixel_delta_u), xadd((double)x, ox))),
                    scale3(ld3(cam.pixel_delta_v), xadd((double)y, oy)));
    d3 ddu = ld3(cam.defocus_disk_u), ddv = ld3(cam.defocus_disk_v);
    bool no_lens = ddu.x == 0.0 && ddu.y == 0.0 && ddu.z == 0.0 && ddv.x == 0.0 && ddv.y == 0.0 && ddv.z == 0.0;
    if (no_lens) {
        o = add3(add3(ld3(cam.look_from), mk3(0.0, 0.0, 0.0)), mk3(0.0, 0.0, 0.0));
    } else {
        d3 p = random_in_unit_disk(s);
        o = add3(add3(ld3(cam.look_from), scale3(ddu, p.x)), scale3(ddv, p.y));
    }
    d = sub3(point, o);
}
