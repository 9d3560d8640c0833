// pool_kernel.cuh — the pooled persistent render kernel (sm_100a).  Included by nrrt_device.cu.
//
// Why: with one path per lane, a warp's lanes sit in different stages of Camera::get_ray_color (walking inner nodes,
// holding a primitive leaf, entering a wrapper, waiting to be shaded) and every stage runs with the few lanes that
// happen to be in it: ncu showed 8 of 32 lanes active in the node loop on the teapot (profiles/r02_*).  Here a warp
// owns a POOL of NS path slots (NS > 32) whose whole state lives in shared memory, lanes own nothing, and the warp
// repeatedly picks the stage with the most ready slots, hands up to 32 of them to its lanes and runs that stage:
//
//   NODE   walk four-slot inner nodes (f32 box filter, rare exact f64 fallback) until the slot holds a leaf
//   PRIM   one exact f64 primitive test (Sphere::hit / Plane::hit), closest-hit update, next stack entry
//   INST   enter a wrapper chain (exact f64 ray transform + nested root box) or leave one (level marker)
//   SHADE  HitRecord + Material::scatter/emit + Texture::get_color, sample accumulation, next camera ray / work item
//
// It is a wavefront renderer whose queues never leave the SM: no ray or hit record round-trips through HBM, no
// inter-warp synchronisation, one launch per image.  Scheduling is warp-synchronous (ballots + a 32-entry
// assignment table), so there are no atomics and no fences on the hot path.  Traversal, intersection and shading
// are the device functions of rt_device.cuh that the other kernel designs use, the work items and Philox counters
// are the same, so the image is bit-identical to theirs.
#pragma once

#ifndef NRRT_POOL_WARPS
#define NRRT_POOL_WARPS 4  // warps per block
#endif
#ifndef NRRT_POOL_NODE_KEEP_NUM
#define NRRT_POOL_NODE_KEEP_NUM 1  // the NODE stage goes on while >= KEEP_NUM/KEEP_DEN of the lanes it started with still
#define NRRT_POOL_NODE_KEEP_DEN 2  // hold an inner node; below that the warp re-schedules (refills the lanes).
                                   // Measured on B200 (teapot / C5 / Cornell, Mrays/s): 7/8 1993 / 1840 / 3682, 3/4 2031 / 1881 /
                                   // 3720, 1/2 2091 / 1949 / 3786.  Slots per warp: 48 1665, 56 1946, 64 2031, 80 1860.
#endif
#define NRRT_POOL_TRIVIAL_MAX 4     // camera rays that miss the scene's root box, absorbed per SHADE visit
#ifndef NRRT_POOL_W_SHADE
#define NRRT_POOL_W_SHADE 8  // stage weights (x/8) of the scheduler's "most ready slots" rule
#endif
#ifndef NRRT_POOL_W_INST
#define NRRT_POOL_W_INST 8
#endif
#ifndef NRRT_POOL_W_PRIM
#define NRRT_POOL_W_PRIM 8
#endif
#ifndef NRRT_POOL_W_NODE
#define NRRT_POOL_W_NODE 8
#endif
#ifndef NRRT_POOL_SCREEN_MIN
#define NRRT_POOL_SCREEN_MIN 8      // NODE stage: lanes holding a plane leaf before the reject-only test runs for them
#endif

enum : uint32_t {
    PS_RETIRED = 0,
    PS_NODE = 1,       // cur = inner node
    PS_PRIM = 2,       // cur = sphere / plane leaf
    PS_INST = 3,       // cur = instance leaf or level marker
    PS_HIT = 4,        // closest-hit query finished: shade it
    PS_NEED_PATH = 5,  // next sample of the slot's work item: Camera::get_ray
    PS_NEED_ITEM = 6   // fetch / decode the next work item
};

// Slot state.  HOT fields — what the traversal stages touch on every visit — live in the warp's shared-memory pool,
// structure of arrays: field k of slot s at base[k * NS + s], so the lanes of a warp (distinct slots) hit distinct
// banks up to the 2-way overlap of slots s and s + 32.  COLD fields — what only the SHADE stage reads (throughput,
// running sum, hit attributes, work-item bookkeeping) and the world-space ray an instance visit has to come back to —
// live in global memory (L2-resident: a few tens of MB for the whole GPU), structure of arrays over all pool slots of
// the launch.  Keeping them out of shared memory is what lets 16 warps x 64 slots fit on an SM instead of 9.
//
// LITE (small scenes, where a closest-hit query is a handful of node visits): two stages only.  TRAVERSE runs the
// lane-owned Traversal of rt_device.cuh to completion for up to 32 ray-ready slots, its working state in registers
// and a per-lane stack; SHADE is the stage above.  A slot then carries only path state, and all of it — the "cold"
// fields too — stays in shared memory (no L2 round trip where shading dominates).
template <uint32_t F, int NS, bool LITE = false>
struct Pool {
    static constexpr bool kInst = (F & NRRT_F_INSTANCES) != 0;
    static constexpr bool kUv = (F & NRRT_F_PLANES) && (F & NRRT_F_TEXTURED);
    static constexpr bool kMotion = (F & NRRT_F_MOTION) != 0;
    // ---- hot doubles: the f64 ray of the slot's CURRENT space (world, or the innermost entered instance's), best t
    static constexpr int D_RAY = 0, D_BT = 6;
    static constexpr int ND = 7;
    // ---- hot words
    static constexpr int W_CTL = 0;     // state[0:4) level[4:7) best_depth[7:10) sp[10:18)
    static constexpr int W_CUR = 1, W_TCULL = 2, W_R32 = 3 /* 7 */, W_BPRIM = 10;
    static constexpr int W_CINST = 11;                         // cur_inst: 4 x u16 in 2 words (kInst)
    static constexpr int W_STACK = W_CINST + (kInst ? 2 : 0);
    static constexpr int W_BPRIM_LITE = 1;                     // LITE: the slot's hot words are CTL and BPRIM only
    static constexpr int NWH = LITE ? 2 : W_STACK;             // hot words before the per-slot stack (full) / cold words (LITE)
    // ---- cold doubles
    static constexpr int C_T = 0, C_SUM = 3, C_P = 6;
    static constexpr int C_AB = 9;                            // alpha, beta (kUv)
    static constexpr int C_DOBJ = C_AB + (kUv ? 2 : 0);       // object-space direction of the best hit (kInst)
    static constexpr int C_WRAY = C_DOBJ + (kInst ? 3 : 0);   // world ray, saved while the slot is inside an instance (kInst, full)
    static constexpr int C_TIME = C_WRAY + ((kInst && !LITE) ? 6 : 0);   // Ray::time (kMotion)
    static constexpr int NCD = C_TIME + (kMotion ? 1 : 0);
    // ---- cold words
    static constexpr int CW_ITEM = 0, CW_SAMPLE = 1, CW_BOUNCE = 2;
    static constexpr int CW_BINST = 3;                        // best.inst: 4 x u16 in 2 words (kInst)
    static constexpr int NCW = CW_BINST + (kInst ? 2 : 0);
    __host__ __device__ static constexpr size_t cold_bytes_per_slot() { return LITE ? 0 : 8 * NCD + 4 * NCW; }
    // Shared memory of one warp.  Full: slots x (hot doubles, hot words, stack of `cap` entries), assignment table.
    // LITE: slots x (hot + cold doubles, hot + cold words), assignment table, and per LANE a stack of `cap` entries and
    // the object-space ray of the instance being traversed.
    static constexpr int kLaneDoubles = (LITE && kInst) ? 6 : 0;
    static constexpr int kAssign = LITE ? ((NS + 31) & ~31) : 32;  // assignment table entries (LITE: every ray-ready slot)
    __host__ __device__ static constexpr size_t bytes_per_warp(uint32_t cap) {
        const size_t b = LITE ? (size_t)NS * (8 * (ND + NCD) + 4 * (NWH + NCW)) + 32 * (8 * kLaneDoubles + 4 * cap) + kAssign * 4
                              : (size_t)NS * (8 * ND + 4 * (W_STACK + cap)) + kAssign * 4;
        return (b + 15) & ~(size_t)15;
    }

    double* D;
    uint32_t* W;
    uint32_t* assign;
    double* lane_d;     // LITE: this lane's object-space ray, lane_d[k * 32]
    uint32_t* lane_stack;  // LITE: this lane's traversal stack, lane_stack[k * 32]
    double* CD;       // cold doubles, already offset to this warp's first slot
    uint32_t* CW;     // cold words, likewise
    size_t cstride;   // pool slots in the launch
    uint32_t cap;     // traversal stack entries per slot
    __device__ __forceinline__ double& d(int k, uint32_t s) const { return D[k * NS + s]; }
    __device__ __forceinline__ uint32_t& w(int k, uint32_t s) const { return W[k * NS + s]; }
    __device__ __forceinline__ double& cd(int k, uint32_t s) const {
        return LITE ? D[(ND + k) * NS + s] : CD[(size_t)k * cstride + s];
    }
    __device__ __forceinline__ uint32_t& cw(int k, uint32_t s) const {
        return LITE ? W[(NWH + k) * NS + s] : CW[(size_t)k * cstride + s];
    }
    __device__ __forceinline__ uint32_t& bprim(uint32_t s) const { return w(LITE ? W_BPRIM_LITE : W_BPRIM, s); }
    __device__ __forceinline__ d3 ld3d(int k, uint32_t s) const { return mk3(d(k, s), d(k + 1, s), d(k + 2, s)); }
    __device__ __forceinline__ void st3d(int k, uint32_t s, d3 v) const { d(k, s) = v.x, d(k + 1, s) = v.y, d(k + 2, s) = v.z; }
    __device__ __forceinline__ d3 ld3c(int k, uint32_t s) const { return mk3(cd(k, s), cd(k + 1, s), cd(k + 2, s)); }
    __device__ __forceinline__ void st3c(int k, uint32_t s, d3 v) const { cd(k, s) = v.x, cd(k + 1, s) = v.y, cd(k + 2, s) = v.z; }
    __device__ __forceinline__ Ray32 ld_r32(uint32_t s) const {
        Ray32 r;
        r.idx = __uint_as_float(w(W_R32, s)), r.idy = __uint_as_float(w(W_R32 + 1, s)), r.idz = __uint_as_float(w(W_R32 + 2, s));
        r.ox = __uint_as_float(w(W_R32 + 3, s)), r.oy = __uint_as_float(w(W_R32 + 4, s)), r.oz = __uint_as_float(w(W_R32 + 5, s));
        r.margin = __uint_as_float(w(W_R32 + 6, s));
        return r;
    }
    __device__ __forceinline__ void st_r32(uint32_t s, const Ray32& r) const {
        w(W_R32, s) = __float_as_uint(r.idx), w(W_R32 + 1, s) = __float_as_uint(r.idy), w(W_R32 + 2, s) = __float_as_uint(r.idz);
        w(W_R32 + 3, s) = __float_as_uint(r.ox), w(W_R32 + 4, s) = __float_as_uint(r.oy), w(W_R32 + 5, s) = __float_as_uint(r.oz);
        w(W_R32 + 6, s) = __float_as_uint(r.margin);
    }
    // the f64 ray of the slot's current space
    __device__ __forceinline__ void ld_ray(uint32_t s, d3& o, d3& dd) const { o = ld3d(D_RAY, s), dd = ld3d(D_RAY + 3, s); }
    __device__ __forceinline__ void st_ray(uint32_t s, d3 o, d3 dd) const { st3d(D_RAY, s, o), st3d(D_RAY + 3, s, dd); }
    // instance chains: four 16-bit instance indices in two words (the render path checks n_instances <= 65536)
    static __device__ __forceinline__ InstChain unpack_chain(uint32_t lo, uint32_t hi) {
        InstChain c;
        c.a = lo & 0xFFFFu, c.b = lo >> 16, c.c = hi & 0xFFFFu, c.d = hi >> 16;
        return c;
    }
    __device__ __forceinline__ InstChain ld_cur_chain(uint32_t s) const { return unpack_chain(w(W_CINST, s), w(W_CINST + 1, s)); }
    __device__ __forceinline__ InstChain ld_best_chain(uint32_t s) const { return unpack_chain(cw(CW_BINST, s), cw(CW_BINST + 1, s)); }
    __device__ __forceinline__ void set_cur_chain(uint32_t s, uint32_t level, uint32_t inst) const {
        uint32_t& wd = w(W_CINST + (level >> 1), s);
        wd = (level & 1u) ? ((wd & 0xFFFFu) | (inst << 16)) : ((wd & 0xFFFF0000u) | inst);
    }
};

__device__ __forceinline__ uint32_t ctl_state(uint32_t c) { return c & 15u; }
__device__ __forceinline__ uint32_t ctl_level(uint32_t c) { return (c >> 4) & 7u; }
__device__ __forceinline__ uint32_t ctl_bdepth(uint32_t c) { return (c >> 7) & 7u; }
__device__ __forceinline__ uint32_t ctl_sp(uint32_t c) { return (c >> 10) & 255u; }
__device__ __forceinline__ uint32_t ctl_make(uint32_t state, uint32_t level, uint32_t bdepth, uint32_t sp) {
    return state | (level << 4) | (bdepth << 7) | (sp << 10);
}
#ifndef NRRT_POOL_PREREJECT
#define NRRT_POOL_PREREJECT 0  // f32 reject-only plane test (plane_prereject) before the exact one:
                               // 0 = off, 1 = inside the NODE stage (a rejected leaf never reaches PRIM), 2 = at the top of PRIM.
                               // Proven sound by the checked build (27 M segments, no hit ever rejected) and measured on B200
                               // (teapot / C5 / Cornell, Mrays/s): off 2116 / 1959 / 3787, NODE stage 2020 / 1779 / 3059,
                               // PRIM stage 2098 / 1887 / 3597 (profiles/r02_pool_variants3.log).  It does not pay: the exact
                               // test already leaves after one dot product and one division when t > best t, the FP64 pipe
                               // is 6 % busy, and what a PRIM visit costs is its scheduling round, not its arithmetic.
#endif
// the stage a slot waits for, from the entry it holds.  With the reject-only plane test a plane leaf first waits for
// the NODE stage (which runs that test) and only one that survived it (`screened`) waits for the PRIM stage.
template <uint32_t F>
__device__ __forceinline__ uint32_t classify_ref(uint32_t cur, bool screened = false) {
    const uint32_t ty = NRRT_REF_TYPE(cur);
    if (ty == NRRT_REF_NODE) return PS_NODE;
    if (ty == NRRT_REF_PLANE) return (NRRT_POOL_PREREJECT == 1 && (F & NRRT_F_PLANES) && !screened) ? PS_NODE : PS_PRIM;
    if (ty == NRRT_REF_SPHERE) return PS_PRIM;
    if (cur == NRRT_REF_NONE) return PS_HIT;
    return PS_INST;  // instance leaf or NRRT_REF_POP
}

// ---- start of a closest-hit query (Traversal::begin on pool state): returns the first entry
template <uint32_t F, int NS, bool LITE>
__device__ __forceinline__ uint32_t pool_begin(const DevScene& S, const Pool<F, NS, LITE>& P, uint32_t s, d3 wo, d3 wd) {
    using PL = Pool<F, NS, LITE>;
    const double tmin = 0.001, tmax = NRRT_INF;
    const float tmin32 = (float)tmin, tmax32 = 3.4e38f;
    const Ray32 r32 = make_ray32(wo, wd);
    P.st_r32(s, r32);
    P.w(PL::W_TCULL, s) = __float_as_uint(3.4e38f);
    P.d(PL::D_BT, s) = NRRT_INF;
    P.bprim(s) = NRRT_REF_NONE;
    uint32_t cur = S.root;
    if (NRRT_REF_TYPE(cur) == NRRT_REF_NODE) {  // an inner node tests its own box (object.rs:102)
        if (!root_box_test<false>(&S.root_box, r32, wo, wd, tmin, tmax, tmin32, tmax32, nullptr)) cur = NRRT_REF_NONE;
    } else if (cur != NRRT_REF_NONE) {
        // a one-leaf scene: the reference tests no box (object.rs:95-97); cull only what the filter proves missed
        float e, g, m;
        box_filter(r32, (float)S.root_box.lo[0], (float)S.root_box.lo[1], (float)S.root_box.lo[2], (float)S.root_box.hi[0],
                   (float)S.root_box.hi[1], (float)S.root_box.hi[2], tmin32, tmax32, e, g, m);
        if (g < -m) cur = NRRT_REF_NONE;
    }
    return cur;
}

// ---- NODE stage.  A lane walks inner nodes; when it lands on a plane leaf it runs the f32 reject-only test right
// here (plane_prereject) and, if that proves a miss, takes the next stack entry and goes on — four out of five
// primitive tests on a mesh end this way, without a visit to the PRIM stage.
template <uint32_t F, int NS, bool LITE>
__device__ __forceinline__ void pool_node(const DevScene& S, const Pool<F, NS, LITE>& P, uint32_t s, bool valid,
                                          uint32_t n_take) {
    using PL = Pool<F, NS, LITE>;
    constexpr bool kPre = NRRT_POOL_PREREJECT == 1 && (F & NRRT_F_PLANES) != 0;
    const float tmin32 = 0.001f, tmax32 = 3.4e38f;
    uint32_t ctl = 0, cur = NRRT_REF_NONE, sp = 0;
    Ray32 r32{};
    Ray32P rp{};
    float tcull = 0.f;
    if (valid) {
        ctl = P.w(PL::W_CTL, s);
        cur = P.w(PL::W_CUR, s);
        sp = ctl_sp(ctl);
        r32 = P.ld_r32(s);
        tcull = __uint_as_float(P.w(PL::W_TCULL, s));
        if (kPre) {
            d3 o, d;
            P.ld_ray(s, o, d);
            rp = make_ray32p(o, d);
        }
    }
    const uint32_t level = ctl_level(ctl);
    uint32_t* stack = &P.w(PL::W_STACK, s);
    const uint32_t keep = max(1u, (n_take * NRRT_POOL_NODE_KEEP_NUM) / NRRT_POOL_NODE_KEEP_DEN);
    bool tested = false;  // the plane leaf in hand has been through the reject test ("maybe": it needs the exact one)
    for (uint32_t it = 0;; ++it) {
        const bool at_node = valid && NRRT_REF_TYPE(cur) == NRRT_REF_NODE;
        const bool at_plane = kPre && valid && !tested && NRRT_REF_TYPE(cur) == NRRT_REF_PLANE;
        const unsigned m_node = __ballot_sync(0xffffffffu, at_node);
        const unsigned m_plane = kPre ? __ballot_sync(0xffffffffu, at_plane) : 0u;
        const uint32_t n_act = __popc(m_node | m_plane);
        if (n_act == 0 || (it && n_act < keep)) break;
        // one kind of work per trip, chosen for the whole warp: lanes holding a plane leaf wait until enough of them
        // do (or nobody has a node left), so neither code path runs for a lane or two
        const bool screen = kPre && (__popc(m_plane) >= NRRT_POOL_SCREEN_MIN || m_node == 0u);
        if (!screen && at_node) {
            uint32_t nxt[4];
            const uint32_t n = wide_visit<false, false>(
                S, r32, tmin32, tmax32, tcull, NRRT_REF_INDEX(cur), 0.001, NRRT_INF,
                [&](d3& oo, d3& dd) { P.ld_ray(s, oo, dd); }, nullptr, nxt);
            NRRT_CHECK(sp + (n ? n - 1 : 0) <= P.cap, "pool traversal stack overflow");
            if (n > 3) stack[sp * NS] = nxt[3], ++sp;
            if (n > 2) stack[sp * NS] = nxt[2], ++sp;
            if (n > 1) stack[sp * NS] = nxt[1], ++sp;
            cur = nxt[0];
            if (n == 0) {
                cur = NRRT_REF_NONE;
                if (sp) --sp, cur = stack[sp * NS];
            }
        } else if (screen && at_plane) {
            if (plane_prereject(S, NRRT_REF_INDEX(cur), rp, 0.000999f, tcull)) {
#if defined(NRRT_CHECKED) && NRRT_CHECKED
                {   // the reject-only test may only reject what the exact test rejects
                    d3 xo, xd, xp;
                    double xa, xb;
                    P.ld_ray(s, xo, xd);
                    const double xt = plane_t(S, NRRT_REF_INDEX(cur), xo, xd, 0.001, NRRT_INF, P.d(PL::D_BT, s), &xa, &xb, &xp);
                    NRRT_CHECK(!(xt == xt), "plane_prereject rejected a primitive the exact test accepts");
                }
#endif
                cur = NRRT_REF_NONE;
                if (sp) --sp, cur = stack[sp * NS];
            } else {
                tested = true;
            }
        }
    }
    if (valid) {
        P.w(PL::W_CUR, s) = cur;
        P.w(PL::W_CTL, s) = ctl_make(classify_ref<F>(cur, tested), level, ctl_bdepth(ctl), sp);
    }
}

// ---- PRIM stage: one exact primitive test, then the next stack entry
template <uint32_t F, int NS, bool LITE>
__device__ __forceinline__ void pool_prim(const DevScene& S, const Pool<F, NS, LITE>& P, uint32_t s, bool valid) {
    using PL = Pool<F, NS, LITE>;
    if (!valid) return;
    const double tmin = 0.001, tmax = NRRT_INF;
    const uint32_t ctl = P.w(PL::W_CTL, s);
    const uint32_t leaf = P.w(PL::W_CUR, s);
    const uint32_t level = ctl_level(ctl);
    uint32_t sp = ctl_sp(ctl), bdepth = ctl_bdepth(ctl);
    d3 o, d;
    P.ld_ray(s, o, d);
    const double best_t = P.d(PL::D_BT, s);
    double a_ = 0.0, b_ = 0.0, t;
    d3 pt;
    if ((F & NRRT_F_SPHERES) && (!(F & NRRT_F_PLANES) || NRRT_REF_TYPE(leaf) == NRRT_REF_SPHERE)) {
        t = sphere_t<F>(S, NRRT_REF_INDEX(leaf), o, d, tmin, tmax, PL::kMotion ? P.cd(PL::C_TIME, s) : 0.0);
        pt = ray_at(o, d, t);
    } else if (NRRT_POOL_PREREJECT == 2 &&
               plane_prereject(S, NRRT_REF_INDEX(leaf), make_ray32p(o, d), 0.000999f, __uint_as_float(P.w(PL::W_TCULL, s)))) {
        t = __longlong_as_double(0x7ff8000000000000LL);  // proven miss: the exact test would return None
#if defined(NRRT_CHECKED) && NRRT_CHECKED
        const double xt = plane_t(S, NRRT_REF_INDEX(leaf), o, d, tmin, tmax, best_t, &a_, &b_, &pt);
        NRRT_CHECK(!(xt == xt), "plane_prereject rejected a primitive the exact test accepts");
#endif
    } else {
        t = plane_t(S, NRRT_REF_INDEX(leaf), o, d, tmin, tmax, best_t, &a_, &b_, &pt);
    }
    if (t == t) {
        bool take = t < best_t;
        if (!take && t == best_t) {
            InstChain cc, bc;
            cc.clear(), bc.clear();
            if (PL::kInst) cc = P.ld_cur_chain(s), bc = P.ld_best_chain(s);
            take = tie_candidate_wins(S, leaf, cc, level, bc, P.bprim(s), bdepth);
        }
        if (take) {
            P.d(PL::D_BT, s) = t;
            P.bprim(s) = leaf;
            bdepth = level;
            if (PL::kInst && level) {
                P.cw(PL::CW_BINST, s) = P.w(PL::W_CINST, s), P.cw(PL::CW_BINST + 1, s) = P.w(PL::W_CINST + 1, s);
                P.st3c(PL::C_DOBJ, s, d);
            }
            P.st3c(PL::C_P, s, pt);
            if (PL::kUv) P.cd(PL::C_AB, s) = a_, P.cd(PL::C_AB + 1, s) = b_;
            const float tf = (float)t;  // f32 upper bound of t with slack far above any f64 rounding discrepancy
            P.w(PL::W_TCULL, s) = __float_as_uint(tf + fabsf(tf) * 1.0e-6f + 1e-30f);
        }
    }
    uint32_t cur = NRRT_REF_NONE;
    if (sp) --sp, cur = P.w(PL::W_STACK + sp, s);
    P.w(PL::W_CUR, s) = cur;
    P.w(PL::W_CTL, s) = ctl_make(classify_ref<F>(cur), level, bdepth, sp);
}

// ---- INST stage: enter a wrapper chain, or leave one (level marker)
template <uint32_t F, int NS, bool LITE>
__device__ __forceinline__ void pool_inst(const DevScene& S, const Pool<F, NS, LITE>& P, uint32_t s, bool valid) {
    using PL = Pool<F, NS, LITE>;
    if (!PL::kInst || !valid) return;
    const double tmin = 0.001, tmax = NRRT_INF;
    const float tmin32 = 0.001f, tmax32 = 3.4e38f;
    const uint32_t ctl = P.w(PL::W_CTL, s);
    uint32_t cur = P.w(PL::W_CUR, s), level = ctl_level(ctl), sp = ctl_sp(ctl);
    if (cur == NRRT_REF_POP) {
        // leaving an instance: rebuild the parent level's ray from the world ray (bit-identical recomputation)
        --level;
        d3 po = P.ld3c(PL::C_WRAY, s), pd = P.ld3c(PL::C_WRAY + 3, s);
        if (level) {
            const InstChain cc = P.ld_cur_chain(s);
#pragma unroll
            for (int l = 0; l < NRRT_MAX_INSTANCE_DEPTH; ++l)
                if (l < (int)level) instance_ray(S, cc.get(l), po, pd);
        }
        P.st_ray(s, po, pd);
        P.st_r32(s, make_ray32(po, pd));
    } else {
        const uint32_t ii = NRRT_REF_INDEX(cur);
        const nrrt_instance* in = &S.instances[ii];
        const uint32_t inner = in->inner;
        if (inner != NRRT_REF_NONE && level < NRRT_MAX_INSTANCE_DEPTH) {
            d3 no, nd;
            P.ld_ray(s, no, nd);
            const d3 wo = no, wd = nd;
            instance_ray_inl(S, ii, no, nd);
            const Ray32 n32 = make_ray32(no, nd);
            bool enter = true;
            if (NRRT_REF_TYPE(inner) == NRRT_REF_NODE)
                enter = root_box_test<false>(&in->inner_box, n32, no, nd, tmin, tmax, tmin32, tmax32, nullptr);
            if (enter) {
                if (level == 0) P.st3c(PL::C_WRAY, s, wo), P.st3c(PL::C_WRAY + 3, s, wd);  // the way back to world space
                NRRT_CHECK(sp < P.cap, "pool traversal stack overflow (level marker)");
                P.w(PL::W_STACK + sp, s) = NRRT_REF_POP;
                ++sp;
                P.set_cur_chain(s, level, ii);
                ++level;
                P.st_ray(s, no, nd);
                P.st_r32(s, n32);
                P.w(PL::W_CUR, s) = inner;
                P.w(PL::W_CTL, s) = ctl_make(classify_ref<F>(inner), level, ctl_bdepth(ctl), sp);
                return;
            }
        }
    }
    cur = NRRT_REF_NONE;
    if (sp) --sp, cur = P.w(PL::W_STACK + sp, s);
    P.w(PL::W_CUR, s) = cur;
    P.w(PL::W_CTL, s) = ctl_make(classify_ref<F>(cur), level, ctl_bdepth(ctl), sp);
}

// ---- TRAVERSE stage (LITE): whole closest-hit queries, lane-owned traversal state
// Per-query context of Traversal (rt_device.cuh): world ray from the slot, object-space ray in the lane's scratch,
// attributes of a new best hit straight into the slot.
template <uint32_t F, int NS>
struct PoolLiteCtx {
    static constexpr bool kRayInCtx = true;
    using PL = Pool<F, NS, true>;
    const PL& P;
    uint32_t s;
    __device__ __forceinline__ double time() const { return PL::kMotion ? P.cd(PL::C_TIME, s) : 0.0; }
    __device__ __forceinline__ void get(d3& oo, d3& dd) const { P.ld_ray(s, oo, dd); }
    __device__ __forceinline__ void get_obj(d3& oo, d3& dd) const {
        const double* q = P.lane_d;
        oo = mk3(q[0], q[32], q[64]), dd = mk3(q[96], q[128], q[160]);
    }
    __device__ __forceinline__ void put_obj(d3 oo, d3 dd) const {
        double* q = P.lane_d;
        q[0] = oo.x, q[32] = oo.y, q[64] = oo.z, q[96] = dd.x, q[128] = dd.y, q[160] = dd.z;
    }
    __device__ __forceinline__ void put(uint32_t level, d3 p, double a, double b, d3 dobj) const {
        P.st3c(PL::C_P, s, p);
        if (PL::kUv) P.cd(PL::C_AB, s) = a, P.cd(PL::C_AB + 1, s) = b;
        if (PL::kInst && level) P.st3c(PL::C_DOBJ, s, dobj);
    }
};
// WIDE: walk the four-slot nodes, or the binary ones (what the small scenes this variant serves are uploaded with too).
// The assignment table holds ALL n_ready ray-ready slots of the pool (up to NS): the lanes start with the first 32 and,
// whenever NRRT_POOL_REFILL_MIN of them have finished their query, the idle lanes take the next slots from the table
// — queries differ in length (an instance entry, a deeper subtree), and without the refill the stage ran with 11 of
// 32 lanes while it waited for the longest one.
#ifndef NRRT_POOL_REFILL_MIN
#define NRRT_POOL_REFILL_MIN 8
#endif
template <uint32_t F, int NS, bool WIDE>
__device__ __forceinline__ void pool_traverse(const DevScene& S, const Pool<F, NS, true>& P, uint32_t n_ready) {
    using PL = Pool<F, NS, true>;
    const uint32_t lane = threadIdx.x & 31u;
    Traversal<false, false, F, false, WIDE> tr;
    uint32_t s = 0, next = 0;
    bool running = false;
    for (;;) {
        const unsigned idle = __ballot_sync(0xffffffffu, !running);
        if (next < n_ready && (idle == 0xffffffffu || __popc(idle) >= NRRT_POOL_REFILL_MIN)) {
            const uint32_t mine = next + __popc(idle & ((1u << lane) - 1u));
            if (!running && mine < n_ready) {
                s = P.assign[mine];
                NRRT_CHECK(s < NS && ctl_state(P.w(PL::W_CTL, s)) == PS_NODE, "TRAVERSE: slot is not ray-ready");
                tr.begin(S, PoolLiteCtx<F, NS>{P, s}, 0.001, NRRT_INF, nullptr);
                running = true;
            }
            next += __popc(idle);
        }
        if (!__any_sync(0xffffffffu, running)) break;
        if (tr.round(S, PoolLiteCtx<F, NS>{P, s}, 0.001, NRRT_INF, P.lane_stack, 32, nullptr, running) && running) {
            P.d(PL::D_BT, s) = tr.best.t;
            P.bprim(s) = tr.best.prim;
            if (PL::kInst && tr.best.depth) {
                P.cw(PL::CW_BINST, s) = tr.best.inst.a | (tr.best.inst.b << 16);
                P.cw(PL::CW_BINST + 1, s) = tr.best.inst.c | (tr.best.inst.d << 16);
            }
            P.w(PL::W_CTL, s) = ctl_make(PS_HIT, 0, tr.best.depth, 0);
            running = false;
        }
    }
}

// ---- SHADE stage: shade a finished query, account finished paths, next camera ray / work item, start the next query
template <uint32_t F, int NS, bool LITE>
__device__ __forceinline__ void pool_shade(const DevScene& S, const nrrt_camera& cam, const RenderParams& RP,
                                           const Pool<F, NS, LITE>& P, uint32_t s, bool valid, double* __restrict__ partials,
                                           unsigned long long* __restrict__ counters, uint32_t& segs, uint32_t& paths,
                                           uint32_t& wb_next, uint32_t& wb_end) {
    using PL = Pool<F, NS, LITE>;
    // (called by all 32 lanes: the work-item fetch in the middle is a warp operation; lanes without a slot skip the rest)
    const uint32_t ctl = valid ? P.w(PL::W_CTL, s) : ctl_make(PS_RETIRED, 0, 0, 0);
    uint32_t state = ctl_state(ctl);
    uint32_t item = valid ? P.cw(PL::CW_ITEM, s) : 0u;
    WorkItem wi;
    wi.x = wi.y = wi.sample_end = 0;
    Sampler smp{RP.key, 0u, 0u};
    if (valid && state != PS_NEED_ITEM) {
        decode_item<(F & NRRT_F_ACTIVE) != 0>(cam, RP, item, wi);
        smp.pixel = wi.y * cam.width + wi.x;
        smp.sample = P.cw(PL::CW_SAMPLE, s);
    }
    uint32_t bounce = valid ? P.cw(PL::CW_BOUNCE, s) : 0u;
    d3 o = mk3(0, 0, 0), d = o;
    bool start = false;  // a new closest-hit query starts from (o, d)
    if (state == PS_HIT) {
        P.ld_ray(s, o, d);  // the stack is empty, so every level marker has been consumed: this is the world ray
        d3 T = P.ld3c(PL::C_T, s);
        d3 L = mk3(0.0, 0.0, 0.0);
        bool alive;
        HitId h;
        h.prim = P.bprim(s);
        if (h.prim == NRRT_REF_NONE) {  // camera.rs:298
            L = mul3(T, ld3(cam.background));
            alive = false;
        } else {
            h.t = P.d(PL::D_BT, s);
            h.depth = ctl_bdepth(ctl);
            h.inst.clear();
            if (PL::kInst && h.depth) h.inst = P.ld_best_chain(s);
            HitRec rec;
            const d3 p_obj = P.ld3c(PL::C_P, s);
            d3 d_dir = d;
            if (PL::kInst && h.depth) d_dir = P.ld3c(PL::C_DOBJ, s);
            double al = 0.0, be = 0.0;
            if (PL::kUv) al = P.cd(PL::C_AB, s), be = P.cd(PL::C_AB + 1, s);
            const bool want_uv = (F & NRRT_F_TEXTURED) && (S.material_flags[hit_material<F>(S, h.prim)] & 1u) != 0;
            resolve_hit_attr<F>(S, h, p_obj, al, be, d_dir, PL::kMotion ? P.cd(PL::C_TIME, s) : 0.0, want_uv, rec);
            alive = path_shade<F>(S, cam, rec, smp, o, d, T, L, bounce);
        }
        if (alive) {
            P.st_ray(s, o, d), P.st3c(PL::C_T, s, T);
            start = true;
        } else {  // path finished: add it to the item's partial sum (sample order)
            const d3 sum = add3(P.ld3c(PL::C_SUM, s), L);
            ++smp.sample;
            if (smp.sample >= wi.sample_end) {  // item finished: publish, fetch the next one
                const size_t pb = (size_t)item * 3;
                partials[pb] = sum.x, partials[pb + 1] = sum.y, partials[pb + 2] = sum.z;
                item = NRRT_NO_ITEM;  // fetched below, by the warp
                state = PS_NEED_ITEM;
            } else {
                P.st3c(PL::C_SUM, s, sum);
                state = PS_NEED_PATH;
            }
        }
    }
    // Work items come to the WARP in blocks of NRRT_ITEM_BLOCK consecutive ones (= consecutive pixels of one chunk), so
    // the slots of a pool stay on neighbouring pixels however far they drift apart in time; one atomic per block.
    {
        const bool want = state == PS_NEED_ITEM && item == NRRT_NO_ITEM;
        const unsigned need = __ballot_sync(0xffffffffu, want);
        if (need) {
            const uint32_t lane = threadIdx.x & 31u, n = __popc(need), rank = __popc(need & ((1u << lane) - 1u));
            const uint32_t avail = wb_end - wb_next;
            uint32_t fresh_base = 0, fresh_size = 0;
            if (n > avail) {
                const uint32_t leader = __ffs(need) - 1;
                if (lane == leader) {
                    fresh_size = item_block_size(RP, *(volatile unsigned long long*)&counters[5], n - avail);
                    fresh_base = (uint32_t)atomicAdd(&counters[5], (unsigned long long)fresh_size);
                }
                fresh_base = __shfl_sync(0xffffffffu, fresh_base, leader);
                fresh_size = __shfl_sync(0xffffffffu, fresh_size, leader);
            }
            if (want) item = rank < avail ? wb_next + rank : fresh_base + (rank - avail);
            if (n > avail) wb_next = fresh_base + (n - avail), wb_end = fresh_base + fresh_size;
            else wb_next += n;
        }
    }
    if (!valid) return;
    if (state == PS_NEED_ITEM) {
        if (item >= RP.n_items) {
            P.cw(PL::CW_ITEM, s) = item;
            P.w(PL::W_CTL, s) = ctl_make(PS_RETIRED, 0, 0, 0);
            return;
        }
        smp.sample = decode_item<(F & NRRT_F_ACTIVE) != 0>(cam, RP, item, wi);
        smp.pixel = wi.y * cam.width + wi.x;
        P.st3c(PL::C_SUM, s, mk3(0.0, 0.0, 0.0));
        state = PS_NEED_PATH;
    }
    uint32_t cur = NRRT_REF_NONE;
    for (int rep = 0;; ++rep) {
        if (state == PS_NEED_PATH) {  // Camera::get_ray for the item's next sample
            double tm;
            camera_ray<PL::kMotion>(cam, wi.x, wi.y, smp, o, d, tm);
            if (PL::kMotion) P.cd(PL::C_TIME, s) = tm;
            P.st_ray(s, o, d), P.st3c(PL::C_T, s, mk3(1.0, 1.0, 1.0));
            bounce = 0;
            ++paths;
            start = true;
        }
        if (!start) break;
        ++segs;
        if (LITE) {  // the TRAVERSE stage starts the query itself
            state = PS_NODE;
            break;
        }
        cur = pool_begin<F, NS, LITE>(S, P, s, o, d);
        state = classify_ref<F>(cur);
        // A camera ray that misses the scene's root box is a finished path on the spot (every other camera ray of an
        // object in front of a background): account for it here instead of spending another SHADE visit on it.
        if (cur != NRRT_REF_NONE || bounce != 0 || rep >= NRRT_POOL_TRIVIAL_MAX) break;
        const d3 sum = add3(P.ld3c(PL::C_SUM, s), ld3(cam.background));  // T = (1,1,1): 1*bg is exact, camera.rs:298
        ++smp.sample;
        start = false;
        if (smp.sample >= wi.sample_end) {
            const size_t pb = (size_t)item * 3;
            partials[pb] = sum.x, partials[pb + 1] = sum.y, partials[pb + 2] = sum.z;
            item = NRRT_NO_ITEM;
            state = PS_NEED_ITEM;  // the next SHADE visit fetches and decodes one
            break;
        }
        P.st3c(PL::C_SUM, s, sum);
        state = PS_NEED_PATH;
    }
    P.cw(PL::CW_ITEM, s) = item;
    P.cw(PL::CW_SAMPLE, s) = smp.sample;
    P.cw(PL::CW_BOUNCE, s) = bounce;
    if (!LITE) P.w(PL::W_CUR, s) = cur;
    P.w(PL::W_CTL, s) = ctl_make(state, 0, 0, 0);
}

// counters: [0]=segments [1]=paths [5]=next work item
// blockDim.x = 32 * (warps per block, <= NRRT_POOL_WARPS), dynamic shared memory = warps * bytes_per_warp(stack_cap)
// cold = the cold slot state of the whole launch: cold_slots x NCD doubles, then cold_slots x NCW words.
#ifndef NRRT_POOL_MIN_BLOCKS
#define NRRT_POOL_MIN_BLOCKS 4  // resident blocks per SM the kernel is compiled for (register budget 65536 / (MB * 128))
#endif
template <uint32_t F, int NS, bool LITE>
__global__ void __launch_bounds__(NRRT_POOL_WARPS * 32, NRRT_POOL_MIN_BLOCKS)
k_render_pool(const __grid_constant__ DevScene S, const __grid_constant__ nrrt_camera cam,
              const __grid_constant__ RenderParams RP, double* __restrict__ partials,
              unsigned long long* __restrict__ counters, uint32_t stack_cap, double* __restrict__ cold,
              uint32_t cold_slots) {
    using PL = Pool<F, NS, LITE>;
    extern __shared__ __align__(16) unsigned char s_pool[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    unsigned char* base = s_pool + (size_t)warp * PL::bytes_per_warp(stack_cap);
    PL P;
    P.D = reinterpret_cast<double*>(base);
    if (LITE) {  // doubles: slots x (hot + cold), lanes x object-space ray; words: slots x (hot + cold), assignment, lane stacks
        P.lane_d = P.D + (size_t)NS * (PL::ND + PL::NCD) + lane;
        P.W = reinterpret_cast<uint32_t*>(P.D + (size_t)NS * (PL::ND + PL::NCD) + 32 * PL::kLaneDoubles);
        P.assign = P.W + (size_t)NS * (PL::NWH + PL::NCW);
        P.lane_stack = P.assign + PL::kAssign + lane;
    } else {
        P.lane_d = nullptr, P.lane_stack = nullptr;
        P.W = reinterpret_cast<uint32_t*>(base + (size_t)NS * 8 * PL::ND);
        P.assign = P.W + (size_t)NS * (PL::W_STACK + stack_cap);
    }
    const uint32_t gwarp = blockIdx.x * (blockDim.x >> 5) + warp;
    P.cstride = cold_slots;
    P.cap = stack_cap;
    NRRT_CHECK(LITE || (size_t)(gwarp + 1) * NS <= cold_slots, "cold state index");
    P.CD = cold + (size_t)gwarp * NS;
    P.CW = reinterpret_cast<uint32_t*>(cold + (size_t)PL::NCD * cold_slots) + (size_t)gwarp * NS;
    uint32_t segs = 0, paths = 0;
    uint32_t wb_next = 0, wb_end = 0;  // this warp's block of work items (warp-uniform)
    // the first n_slots items are pre-assigned (slot k of the grid takes item k); the counter starts at n_slots
    for (uint32_t s = lane; s < NS; s += 32) {
        const uint32_t item = gwarp * NS + s;
        P.cw(PL::CW_ITEM, s) = item;
        P.cw(PL::CW_SAMPLE, s) = 0;
        P.cw(PL::CW_BOUNCE, s) = 0;
        if (!LITE) P.w(PL::W_CUR, s) = NRRT_REF_NONE;
        P.w(PL::W_CTL, s) = ctl_make(item < RP.n_slots ? PS_NEED_ITEM : PS_RETIRED, 0, 0, 0);
    }
    constexpr int NSET = (NS + 31) / 32;  // slots a lane inspects when scheduling
    for (;;) {
        __syncwarp();
        // ---- schedule: count the slots waiting for each stage
        // (one warp reduction over per-stage byte counters: stage k adds 1 << 8k; NS < 256)
        uint32_t st[NSET], packed = 0;
#pragma unroll
        for (int j = 0; j < NSET; ++j) {
            const uint32_t s = lane + 32 * j;
            st[j] = (s < NS) ? ctl_state(P.w(PL::W_CTL, s)) : PS_RETIRED;
            if (st[j] != PS_RETIRED) packed += 1u << (8u * (min(st[j], (uint32_t)PS_HIT) - 1u));
        }
        packed = __reduce_add_sync(0xffffffffu, packed);
        const uint32_t cnt[4] = {packed & 255u, (packed >> 8) & 255u, (packed >> 16) & 255u, packed >> 24};  // NODE PRIM INST SHADE
        if (packed == 0) break;
        // the stage with the most ready slots (ties: later stages first — they free slots for new rays)
        // (a stage's count is weighed by NRRT_POOL_W_* / 8 before the comparison: a long stage is worth running only
        // with more lanes; a stage with nothing ready never wins)
        uint32_t phase = 3, best = cnt[3], score = cnt[3] * NRRT_POOL_W_SHADE;
        if (cnt[2] * NRRT_POOL_W_INST > score) phase = 2, best = cnt[2], score = cnt[2] * NRRT_POOL_W_INST;
        if (cnt[1] * NRRT_POOL_W_PRIM > score) phase = 1, best = cnt[1], score = cnt[1] * NRRT_POOL_W_PRIM;
        if (cnt[0] * NRRT_POOL_W_NODE > score) phase = 0, best = cnt[0], score = cnt[0] * NRRT_POOL_W_NODE;
        if (LITE) {
            // two stages: drain SHADE completely, then TRAVERSE finds EVERY live slot ray-ready and works through them
            // 32 at a time with in-stage refill — the long queries of one batch overlap the short ones of the next
            phase = cnt[3] ? 3u : 0u;
            best = cnt[3] ? cnt[3] : cnt[0];
        }
        // ---- hand the first min(32, best) ready slots to the lanes
        uint32_t rank = 0;
#pragma unroll
        for (int j = 0; j < NSET; ++j) {
            const bool mine = phase == 3 ? st[j] >= PS_HIT : st[j] == phase + 1;
            const unsigned m = __ballot_sync(0xffffffffu, mine);
            const uint32_t r = rank + __popc(m & ((1u << lane) - 1u));
            if (mine && r < (uint32_t)((LITE && phase == 0) ? PL::kAssign : 32)) P.assign[r] = lane + 32 * j;
            rank += __popc(m);
        }
        __syncwarp();
        const uint32_t n_take = min(best, 32u);
        const bool valid = lane < n_take;
        const uint32_t s = valid ? P.assign[lane] : 0u;
        NRRT_CHECK(s < NS, "pool slot index");
        NRRT_CHECK(!valid || (phase == 3 ? ctl_state(P.w(PL::W_CTL, s)) >= PS_HIT : ctl_state(P.w(PL::W_CTL, s)) == phase + 1),
                   "slot handed to the wrong stage");
        __syncwarp();
        if (LITE) {
            if constexpr (LITE) {
                if (phase == 0) pool_traverse<F, NS, false>(S, P, best);
                else pool_shade<F, NS, true>(S, cam, RP, P, s, valid, partials, counters, segs, paths, wb_next, wb_end);
            }
        } else if constexpr (!LITE) {
            if (phase == 0) pool_node<F, NS, false>(S, P, s, valid, n_take);
            else if (phase == 1) pool_prim<F, NS, false>(S, P, s, valid);
            else if (phase == 2) pool_inst<F, NS, false>(S, P, s, valid);
            else pool_shade<F, NS, false>(S, cam, RP, P, s, valid, partials, counters, segs, paths, wb_next, wb_end);
        }
    }
    // block-level reduction of the counters
    __shared__ unsigned long long s_cnt[2];
    if (threadIdx.x == 0) s_cnt[0] = s_cnt[1] = 0;
    __syncthreads();
    unsigned long long segs64 = segs, paths64 = paths;
    for (int off = 16; off; off >>= 1) {
        segs64 += __shfl_down_sync(0xffffffffu, segs64, off);
        paths64 += __shfl_down_sync(0xffffffffu, paths64, off);
    }
    if (lane == 0) {
        atomicAdd(&s_cnt[0], segs64);
        atomicAdd(&s_cnt[1], paths64);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicAdd(&counters[0], s_cnt[0]);
        atomicAdd(&counters[1], s_cnt[1]);
    }
}
