// nrrt_device.cu — CUDA kernels (sm_100a) and the device half of the C ABI (include/nrrt.h).
//
// Kernels
//   k_trace_rays      BVH::hit for a batch of fixed rays (known-answer tests, traversal microbenchmark)
//   k_render_mega     persistent per-thread path loop: camera ray -> (closest hit -> shade/scatter)* with
//                     in-lane path regeneration; state lives in registers
//   k_wf_init/extend/shade   wavefront variant: ray-gen, traverse/intersect and shade/scatter(+regeneration,
//                     +warp-ballot queue compaction) as separate kernels over SoA path state in HBM
//   k_resolve         per-pixel sample accumulation -> f32 RGB (camera.rs:329-337)
// There is no CPU fallback: every entry point fails with NRRT_ERR_NO_DEVICE / NRRT_ERR_CUDA when the GPU
// is unavailable.

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <chrono>
#include <vector>

#include "rt_device.cuh"

#define NRRT_BLOCK 128
#define NRRT_NO_ITEM 0xFFFFFFFFu
#ifndef NRRT_ITEM_BLOCK
#define NRRT_ITEM_BLOCK 128  // work items a warp takes from the global counter at a time (at most)
#endif
#ifndef NRRT_SPLIT_QUEUE
#define NRRT_SPLIT_QUEUE 0  // 1: camera rays and bounce rays occupy separate regions of the ray queue.
// Measured on B200 (round 1): splitting is 3.4x SLOWER (Cornell 3439 -> 994 Mseg/s, earth 4941 -> 1263).  With one
// queue every slot survives every pass (in-slot regeneration), so the queue stays in near-ascending slot order and
// the SoA path state is read and written coalesced; splitting it re-partitions the order every pass until the 32
// slots of a warp are scattered and each 8-byte access costs a 32-byte sector.  Kept as a switch for the record.
#endif

// =========================================================================== kernels
// Work decomposition.  A work item is (owned pixel, sample chunk): the pixel's samples
// [c*chunk, min((c+1)*chunk, spp)).  Items are numbered chunk-major (item = c * n_owned_pixels + pixel) and handed
// out dynamically from one global counter, so every path slot stays busy until the whole image is done no matter
// how uneven the per-pixel path lengths are.  A slot traces its item's samples one after the other, sums their
// radiance in f64 in sample order, writes that partial sum to partials[item] and grabs the next item.
// k_resolve adds a pixel's partials in chunk order: the result does not depend on scheduling, slot count or the
// number of GPUs (chunk size depends on spp only).
// Exact unsigned division by a launch-invariant divisor (round-up multiply-shift, branch free):
// n / d == (t + ((n - t) >> s1)) >> s2 with t = umulhi(m, n).  Replaces three ~20-instruction integer divisions
// per work-item decode.
struct FastDiv {
    uint32_t d, m, s1, s2;
    __host__ static FastDiv make(uint32_t d) {
        FastDiv f;
        f.d = d ? d : 1;
        uint32_t l = 0;
        while ((1ull << l) < f.d) ++l;
        f.m = (uint32_t)(((1ull << 32) * ((1ull << l) - f.d)) / f.d + 1);
        f.s1 = l < 1 ? l : 1;
        f.s2 = l > 0 ? l - 1 : 0;
        return f;
    }
    __host__ __device__ __forceinline__ uint32_t div(uint32_t n) const {
#ifdef __CUDA_ARCH__
        uint32_t t = __umulhi(m, n);
#else
        uint32_t t = (uint32_t)(((uint64_t)m * n) >> 32);
#endif
        return (t + ((n - t) >> s1)) >> s2;
    }
};

struct RenderParams {
    uint2 key;               // Philox key
    uint32_t n_owned_pixels; // pixels rendered by this context
    uint32_t chunk;          // samples of an equal-size work item (the first n_eq chunks of a pixel)
    uint32_t n_eq;           // equal chunks; they cover samples [0, n_eq * chunk)
    uint32_t n_chunks;       // work items per pixel = n_eq + the halving chunks over the remaining samples
    uint32_t c0;             // first chunk of this launch: it renders chunks [c0, c0 + n_items / div_pixels.d)
    uint32_t n_items;        // pixels of the launch * its chunks; items and partials are numbered from c0
    uint32_t long_end;       // item where this launch's equal chunks end (item_block_size)
    uint32_t n_slots;        // paths in flight
    uint32_t n_warps;        // warps that fetch work-item blocks (persistent kernels)
    uint32_t rank, world, rows_per_block;
    FastDiv div_pixels, div_rows;  // by the pixels of the launch (n_owned_pixels, or the active ones), rows_per_block
    FastDiv div_tile, div_strip, div_last;  // by tile_rows, by width * tile_rows (pixels of a full strip), by the rows of the last strip
    uint32_t full_strips;          // strips of tile_rows owned rows
    // adaptive pass: the launch's pixels are active[0 .. div_pixels.d), owned-pixel indices in ascending order
    // (null: every owned pixel, div_pixels.d = n_owned_pixels)
    const uint32_t* active;
};

// owned pixel index -> (x, y) and the owned row j: rank owns row-blocks b with b % world == rank.
// Owned pixels are numbered in STRIPS of tile_rows owned rows, column by column inside a strip, so that a run of
// consecutive indices — the block of work items a warp takes (NRRT_ITEM_BLOCK = 128) — is a compact tile of the image
// (16 columns x 8 rows on one GPU): rays of neighbouring lanes see the same part of the tree and the same materials.
// tile_rows = the largest divisor of rows_per_block up to NRRT_TILE_ROWS, so a tile never straddles two row-blocks —
// which in a shared image lie `world` blocks apart (measured at N = 8 with single-row blocks and 8-row tiles: a tile
// stretched over 64 image rows and the render lost all the coherence gain).  With single rows the tile is a 128-pixel
// piece of one row, which is nearly as good (Cornell -0.4 %, teapot -1.8 % on one GPU).  The last strip may be shorter.
#ifndef NRRT_TILE_ROWS
#define NRRT_TILE_ROWS 8
#endif
__host__ __device__ __forceinline__ void owned_pixel(const nrrt_camera& cam, const RenderParams& P, uint32_t po, uint32_t& x,
                                            uint32_t& y, uint32_t& j) {
    const uint32_t strip = P.div_strip.div(po), k = po - strip * P.div_strip.d;  // div_strip.d = W * tile_rows
    uint32_t r;
    if (strip < P.full_strips) {
        x = P.div_tile.div(k), r = k - x * P.div_tile.d;
    } else {
        x = P.div_last.div(k), r = k - x * P.div_last.d;  // the cut-off last strip: div_last.d rows
    }
    j = strip * P.div_tile.d + r;
    const uint32_t b = P.div_rows.div(j), rr = j - b * P.rows_per_block;
    y = (b * P.world + P.rank) * P.rows_per_block + rr;
}

// Size of the next block of work items a warp takes: NRRT_ITEM_BLOCK while work is plentiful, shrinking to 32 (one per
// lane) as the image runs out — so that the render does not end with a few warps still holding four items per lane
// (a 400x225 image is 9 ms of work: blocks of 128 to the end cost it 20 %).  `next` is the global counter as last seen.
// Items are chunk-major and the equal chunks come first: the LONG items end at item long_end, and a warp
// that has just taken 128 of them when they run out keeps the GPU waiting for 4 long items per lane while everyone
// else is through the short tail chunks — so the blocks also shrink towards that point (measured at N = 8, where a
// GPU has 130 ms of work: 7 ms lost without this).
__device__ __forceinline__ uint32_t item_block_size(const RenderParams& P, unsigned long long next, uint32_t need) {
    const uint32_t end = next < P.long_end ? P.long_end : P.n_items;
    const uint32_t left = next < end ? end - (uint32_t)next : 0u;
    uint32_t b = left / (2u * max(P.n_warps, 1u));
    b = min(max(b, 32u), (uint32_t)NRRT_ITEM_BLOCK);
    return max(b, need);
}

struct WorkItem {
    uint32_t x, y;        // pixel
    uint32_t sample_end;  // one past the last sample of the chunk
};
// item -> pixel + sample range; returns the first sample.  The chunk c is absolute (the launch's item 0 is chunk c0's
// first pixel), so a pixel's samples and their Philox counters do not depend on which launch renders them.
// ACTIVE: an adaptive pass (P.active set), whose item's pixel is the po-th active one.  A compile-time flag, so that
// the kernels of a plain render carry no trace of the list: tested at run time, the load is predicated rather than
// branched around and the benchmark's one-shot render lost 0.5 % to it (measured on B200).
template <bool ACTIVE = false>
__host__ __device__ __forceinline__ uint32_t decode_item(const nrrt_camera& cam, const RenderParams& P, uint32_t item,
                                                         WorkItem& wi) {
    uint32_t c = P.div_pixels.div(item), po = item - c * (ACTIVE ? P.div_pixels.d : P.n_owned_pixels);
    c += P.c0;
    if (ACTIVE) {
#ifdef __CUDA_ARCH__
        NRRT_CHECK(P.active && po < P.div_pixels.d, "active[] index");
#endif
        po = P.active[po];
#ifdef __CUDA_ARCH__
        NRRT_CHECK(po < P.n_owned_pixels, "active pixel is not an owned pixel");
#endif
    }
    uint32_t j;
    owned_pixel(cam, P, po, wi.x, wi.y, j);
    const uint32_t spp = cam.samples_per_pixel;
    if (c < P.n_eq) {
        wi.sample_end = (c + 1) * P.chunk;
        return c * P.chunk;
    }
    // the tail of the pixel halves: with R samples left after the equal chunks, tail chunk k covers
    // [base + R - (R >> k), base + R - (R >> (k + 1))), the last one up to spp
    const uint32_t base = P.n_eq * P.chunk, R = spp - base, k = c - P.n_eq;
    wi.sample_end = (c + 1 == P.n_chunks) ? spp : base + R - (R >> (k + 1));
    return base + R - (R >> k);
}

// COMPACT: the closest-hit query alone — 16 bytes out per ray, no HitRecord (traversal microbenchmark)
template <bool VISIT_ALL, bool COUNT, bool COMPACT = false>
__global__ void __launch_bounds__(NRRT_BLOCK)
k_trace_rays(const __grid_constant__ DevScene S, const double* __restrict__ rays, uint64_t n, double tmin, double tmax,
             double time, nrrt_hit* __restrict__ out, unsigned long long* __restrict__ counters) {
    extern __shared__ uint32_t s_stack[];
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n;  // no early return: trace_closest votes across the whole warp
    d3 o = mk3(0.0, 0.0, 0.0), d = mk3(0.0, 0.0, 0.0);
    if (valid) o = ld3(rays + 6 * i), d = ld3(rays + 6 * i + 3);
    HitId h;
    TraceCounters tc{0, 0, 0, 0, 0};
    trace_closest<VISIT_ALL, COUNT>(S, o, d, time, tmin, tmax, s_stack + threadIdx.x, NRRT_BLOCK, h, &tc, valid);
    if (!valid) return;
    if (COMPACT) {
        nrrt_hit_compact c;
        c.t = h.t, c.prim = h.prim, c.depth_inst0 = h.depth | (h.inst.a << 3);
        reinterpret_cast<nrrt_hit_compact*>(out)[i] = c;
        return;
    }
    nrrt_hit r;
    r.t = h.t;
    r.prim = h.prim;
    r.depth = h.depth;
#pragma unroll
    for (int k = 0; k < NRRT_MAX_INSTANCE_DEPTH; ++k) r.inst[k] = h.inst.get(k);
    r._pad = 0;
    if (h.prim != NRRT_REF_NONE) {
        HitRec rec;
        resolve_hit(S, h, o, d, time, true, rec);
        r.point[0] = rec.point.x, r.point[1] = rec.point.y, r.point[2] = rec.point.z;
        r.normal[0] = rec.normal.x, r.normal[1] = rec.normal.y, r.normal[2] = rec.normal.z;
        r.uv[0] = rec.u, r.uv[1] = rec.v;
        r.material = rec.material;
        r.front_face = rec.front_face ? 1u : 0u;
        uint32_t ix = NRRT_REF_INDEX(h.prim);
        r.object = NRRT_REF_TYPE(h.prim) == NRRT_REF_SPHERE ? S.sphere_object[ix] : S.plane_object[ix];
    } else {
        r.point[0] = r.point[1] = r.point[2] = 0.0;
        r.normal[0] = r.normal[1] = r.normal[2] = 0.0;
        r.uv[0] = r.uv[1] = 0.0;
        r.material = 0xFFFFFFFFu;
        r.front_face = 0;
        r.object = 0xFFFFFFFFu;
    }
    out[i] = r;
    if (COUNT) {
        atomicAdd(&counters[0], (unsigned long long)tc.nodes);
        atomicAdd(&counters[1], (unsigned long long)tc.exact);
        atomicAdd(&counters[2], (unsigned long long)tc.prims);
    }
}

// One step of Camera::get_ray_color (camera.rs:269-300) in iterative form:  L += T*emitted; T *= color.
// Returns true while the path is alive.
template <uint32_t F = NRRT_F_ALL>
__device__ __forceinline__ uint32_t hit_material(const DevScene& S, uint32_t prim) {
    if ((F & NRRT_F_SPHERES) && (!(F & NRRT_F_PLANES) || NRRT_REF_TYPE(prim) == NRRT_REF_SPHERE))
        return S.sphere_material[NRRT_REF_INDEX(prim)];
    return S.plane_material[NRRT_REF_INDEX(prim)] & ~NRRT_PLANE_TRIANGLE_BIT;
}
template <uint32_t F = NRRT_F_ALL>
__device__ __forceinline__ bool path_shade(const DevScene& S, const nrrt_camera& cam, const HitRec& rec,
                                           const Sampler& smp, d3& o, d3& d, d3& T, d3& L, uint32_t& bounce) {
    d3 emitted, atten, nd;
    bool cont = shade_hit<F>(S, rec, d, bounce == 0, smp, bounce + 1, emitted, atten, nd);
    L = add3(L, mul3(T, emitted));
    if (!cont) return false;
    T = mul3(T, atten);
    o = rec.point;
    d = nd;
    ++bounce;
    return bounce < cam.ray_max_bounces;  // camera.rs:276-278
}
__device__ __forceinline__ bool path_step(const DevScene& S, const nrrt_camera& cam, const HitId& h, const Sampler& smp,
                                          d3& o, d3& d, double time, d3& T, d3& L, uint32_t& bounce) {
    if (h.prim == NRRT_REF_NONE) {  // camera.rs:298
        L = add3(L, mul3(T, ld3(cam.background)));
        return false;
    }
    HitRec rec;
    resolve_hit(S, h, o, d, time, (S.material_flags[hit_material(S, h.prim)] & 1u) != 0, rec);
    return path_shade(S, cam, rec, smp, o, d, T, L, bounce);
}

// Megakernel variant: persistent threads, whole path state in registers.
//   counters: [0]=segments [1]=paths [2..4]=node/exact/prim counts (COUNT) [5]=next work item
template <bool COUNT, bool ACTIVE>
__global__ void __launch_bounds__(NRRT_BLOCK)
k_render_mega(const __grid_constant__ DevScene S, const __grid_constant__ nrrt_camera cam,
              const __grid_constant__ RenderParams P, double* __restrict__ partials,
              unsigned long long* __restrict__ counters) {
    extern __shared__ uint32_t s_stack[];
    uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long segs = 0, paths = 0;
    TraceCounters tc{0, 0, 0, 0, 0};
    {
        uint32_t item = w;  // the first n_slots items are pre-assigned; the counter starts at n_slots
        WorkItem wi;
        wi.x = wi.y = wi.sample_end = 0;
        Sampler smp{P.key, 0u, 0u};
        d3 sum = mk3(0.0, 0.0, 0.0);
        d3 o = mk3(0.0, 0.0, 0.0), d = o, T = o, L = o;
        double time = 0.0;
        uint32_t bounce = 0;
        bool alive = false, have_item = false;
        bool running = w < P.n_slots;
        while (__any_sync(0xffffffffu, running)) {  // the traversal votes across the warp: keep every lane in the loop
            if (running && !alive) {
                if (!have_item) {
                    if (item >= P.n_items) {
                        running = false;
                    } else {
                        smp.sample = decode_item<ACTIVE>(cam, P, item, wi);
                        smp.pixel = wi.y * cam.width + wi.x;
                        sum = mk3(0.0, 0.0, 0.0);
                        have_item = true;
                    }
                }
                if (running) {
                    camera_ray<true>(cam, wi.x, wi.y, smp, o, d, time);
                    T = mk3(1.0, 1.0, 1.0);
                    L = mk3(0.0, 0.0, 0.0);
                    bounce = 0;
                    alive = true;
                    ++paths;
                }
            }
            HitId h;
            trace_closest<false, COUNT>(S, o, d, time, 0.001, NRRT_INF, s_stack + threadIdx.x, NRRT_BLOCK, h, &tc, running);
            if (running) {
                ++segs;
                alive = path_step(S, cam, h, smp, o, d, time, T, L, bounce);
                if (!alive) {
                    sum = add3(sum, L);
                    if (++smp.sample >= wi.sample_end) {  // chunk done: publish its partial sum, fetch the next item
                        size_t base = (size_t)item * 3;
                        partials[base] = sum.x, partials[base + 1] = sum.y, partials[base + 2] = sum.z;
                        item = (uint32_t)atomicAdd(&counters[5], 1ull);
                        have_item = false;
                    }
                }
            }
        }
    }
    // block-level reduction of the counters
    __shared__ unsigned long long s_cnt[2];
    if (threadIdx.x == 0) s_cnt[0] = s_cnt[1] = 0;
    __syncthreads();
    for (int off = 16; off; off >>= 1) {
        segs += __shfl_down_sync(0xffffffffu, segs, off);
        paths += __shfl_down_sync(0xffffffffu, paths, off);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_cnt[0], segs);
        atomicAdd(&s_cnt[1], paths);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicAdd(&counters[0], s_cnt[0]);
        atomicAdd(&counters[1], s_cnt[1]);
    }
    if (COUNT) {
        atomicAdd(&counters[2], (unsigned long long)tc.nodes);
        atomicAdd(&counters[3], (unsigned long long)tc.exact);
        atomicAdd(&counters[4], (unsigned long long)tc.prims);
        atomicAdd(&counters[6], (unsigned long long)tc.inst);
        atomicAdd(&counters[7], (unsigned long long)tc.inst_miss);
    }
}

// per-pixel sample accumulation: add the launch's n_items / n_owned_pixels chunk partials in chunk order, divide by
// the samples summed, cast to f32 (camera.rs:329-337).  acc (may be null: start from zero) is the pixel's running f64
// sum over earlier chunks, in owned-row order (j, x), and receives the new sum; out (may be null) the image.  A render
// in passes thus makes the one-shot render's additions, in the same order.
__global__ void k_resolve(const __grid_constant__ nrrt_camera cam, const __grid_constant__ RenderParams P,
                          const double* __restrict__ partials, double* __restrict__ acc, double samples,
                          float* __restrict__ out, bool packed) {
    uint32_t po = blockIdx.x * blockDim.x + threadIdx.x;
    if (po >= P.n_owned_pixels) return;
    uint32_t x, y, j;
    owned_pixel(cam, P, po, x, y, j);
    const size_t ab = ((size_t)j * cam.width + x) * 3;
    d3 s = acc ? mk3(acc[ab], acc[ab + 1], acc[ab + 2]) : mk3(0.0, 0.0, 0.0);
    const uint32_t n_chunks = P.n_items / P.n_owned_pixels;
    for (uint32_t c = 0; c < n_chunks; ++c) {
        size_t b = ((size_t)c * P.n_owned_pixels + po) * 3;
        s = add3(s, mk3(partials[b], partials[b + 1], partials[b + 2]));
    }
    if (acc && n_chunks) acc[ab] = s.x, acc[ab + 1] = s.y, acc[ab + 2] = s.z;
    if (!out) return;
    d3 col = div3(s, samples);
    size_t ob = ((size_t)(packed ? j : y) * cam.width + x) * 3;  // packed: the rank's rows in ascending order
    out[ob] = (float)col.x, out[ob + 1] = (float)col.y, out[ob + 2] = (float)col.z;
}

// ---- adaptive sampling (include/nrrt.h).  The test is stated in f64 with every operation rounded on its own, so that
// the host (nrrt_adaptive_converged, compiled with -ffp-contract=off) and a numpy restatement give the device's verdict.
__host__ __device__ __forceinline__ double rn_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ double rn_sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ __forceinline__ double rn_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double rn_div(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
// squared standard error of the mean of one channel, from the chunks as batch means (K >= 2; NaN propagates)
__host__ __device__ __forceinline__ double adaptive_e2(double S, double Q, uint32_t N, uint32_t K) {
    const double n = (double)N, x = rn_sub(Q, rn_div(rn_mul(S, S), n));
    const double d = x < 0.0 ? 0.0 : x;  // rounding can leave Q - S*S/N slightly below zero
    return rn_div(d, rn_mul((double)(K - 1), n));
}
__host__ __device__ __forceinline__ bool adaptive_converged(const double* S, const double* Q, uint32_t N, uint32_t K,
                                                            const nrrt_adaptive_opts& T) {
    if (K < 2 || N < T.min_samples || !(T.rel_error > 0.0 || T.abs_error > 0.0)) return false;
    for (int ch = 0; ch < 3; ++ch) {
        const double m = rn_div(S[ch], (double)N);
        const double tol = rn_add(T.abs_error, rn_mul(T.rel_error, fabs(m)));
        if (!(adaptive_e2(S[ch], Q[ch], N, K) <= rn_mul(tol, tol))) return false;
    }
    return true;
}

// Per-pixel state of an adaptive frame, owned rows packed ([j][x]; S and Q with 3 channels)
struct AdaptiveState {
    double* S;
    double* Q;
    uint32_t* N;
    uint32_t* K;
};

// One thread per active pixel a of a pass over chunks [P.c0, c1): adds the pass's partials (item-indexed: chunk-local
// c * n_active + a) to S and Q in chunk order, sets N and K, and writes keep[a] = the pixel stays active.  S gets the
// additions k_resolve makes, so a pixel that runs every chunk ends on the one-shot sum.
__global__ void k_resolve_adaptive(const __grid_constant__ nrrt_camera cam, const __grid_constant__ RenderParams P,
                                   uint32_t n_active, const double* __restrict__ partials, AdaptiveState A,
                                   const uint32_t* __restrict__ starts, uint32_t c1, nrrt_adaptive_opts T,
                                   uint8_t* __restrict__ keep) {
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_active) return;
    const uint32_t po = P.active[a];
    NRRT_CHECK(po < P.n_owned_pixels, "active pixel is not an owned pixel");
    uint32_t x, y, j;
    owned_pixel(cam, P, po, x, y, j);
    const size_t pix = (size_t)j * cam.width + x;
    NRRT_CHECK(pix < P.n_owned_pixels, "adaptive state index");
    double s[3], q[3];
    for (int ch = 0; ch < 3; ++ch) s[ch] = A.S[3 * pix + ch], q[ch] = A.Q[3 * pix + ch];
    for (uint32_t c = P.c0; c < c1; ++c) {
        const double n_c = (double)(starts[c + 1] - starts[c]);
        const size_t b = ((size_t)(c - P.c0) * n_active + a) * 3;
        for (int ch = 0; ch < 3; ++ch) {
            const double p = partials[b + ch];
            s[ch] = __dadd_rn(s[ch], p);
            q[ch] = __dadd_rn(q[ch], __ddiv_rn(__dmul_rn(p, p), n_c));
        }
    }
    for (int ch = 0; ch < 3; ++ch) A.S[3 * pix + ch] = s[ch], A.Q[3 * pix + ch] = q[ch];
    A.N[pix] = starts[c1];
    A.K[pix] = c1;
    keep[a] = c1 < P.n_chunks && !adaptive_converged(s, q, starts[c1], c1, T);
}

// Ordered compaction of the active list: the kept entries of in[0 .. n), in their order, to out.  Deterministic (no
// atomics), so the next pass's item order is a function of the retired set alone, and ascending stays ascending, so a
// warp's block of items stays a compact tile of the remaining pixels.  (1) a count per block, (2) an exclusive scan of
// the counts in one block, (3) each block scatters its kept entries from its offset on.
#define NRRT_COMPACT_BLOCK 256
__global__ void __launch_bounds__(NRRT_COMPACT_BLOCK) k_compact_count(const uint8_t* __restrict__ keep, uint32_t n,
                                                                      uint32_t* __restrict__ counts) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = __syncthreads_count(i < n && keep[i]);
    if (threadIdx.x == 0) counts[blockIdx.x] = (uint32_t)k;
}
__global__ void __launch_bounds__(1024) k_compact_scan(uint32_t* __restrict__ counts, uint32_t n_blocks,
                                                       uint32_t* __restrict__ total) {
    __shared__ uint32_t s[1024];
    const uint32_t t = threadIdx.x, per = (n_blocks + 1023) / 1024;
    const uint32_t b0 = min(t * per, n_blocks), b1 = min(b0 + per, n_blocks);
    uint32_t mine = 0;
    for (uint32_t b = b0; b < b1; ++b) mine += counts[b];
    s[t] = mine;
    __syncthreads();
    for (uint32_t off = 1; off < 1024; off <<= 1) {  // inclusive scan over the threads' segment sums
        const uint32_t v = t >= off ? s[t - off] : 0u;
        __syncthreads();
        s[t] += v;
        __syncthreads();
    }
    uint32_t run = s[t] - mine;
    for (uint32_t b = b0; b < b1; ++b) {
        const uint32_t cnt = counts[b];
        counts[b] = run;
        run += cnt;
    }
    if (t == 1023) *total = s[t];
}
__global__ void __launch_bounds__(NRRT_COMPACT_BLOCK) k_compact_scatter(const uint32_t* __restrict__ in,
                                                                        const uint8_t* __restrict__ keep, uint32_t n,
                                                                        const uint32_t* __restrict__ offsets,
                                                                        uint32_t* __restrict__ out) {
    __shared__ uint32_t s_warp[NRRT_COMPACT_BLOCK / 32];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool k = i < n && keep[i];
    const uint32_t ballot = __ballot_sync(0xffffffffu, k);
    if (lane == 0) s_warp[warp] = __popc(ballot);
    __syncthreads();
    uint32_t at = offsets[blockIdx.x];
    for (uint32_t w = 0; w < warp; ++w) at += s_warp[w];
    if (k) out[at + __popc(ballot & ((1u << lane) - 1u))] = in[i];
}

// Per-pixel outputs of an adaptive frame, one thread per owned pixel, laid out as k_resolve lays out the image
// (packed: owned rows only).  IMAGE: S / N as f32; ERROR: sqrt(e2) per channel as f32, +inf where K < 2; SAMPLES: N.
enum AdaptiveMap { AMAP_IMAGE, AMAP_ERROR, AMAP_SAMPLES };
template <int WHAT>
__global__ void k_adaptive_map(const __grid_constant__ nrrt_camera cam, const __grid_constant__ RenderParams P,
                               AdaptiveState A, void* __restrict__ out, bool packed) {
    const uint32_t po = blockIdx.x * blockDim.x + threadIdx.x;
    if (po >= P.n_owned_pixels) return;
    uint32_t x, y, j;
    owned_pixel(cam, P, po, x, y, j);
    const size_t pix = (size_t)j * cam.width + x;
    NRRT_CHECK(pix < P.n_owned_pixels, "adaptive state index");
    const size_t ob = (size_t)(packed ? j : y) * cam.width + x;
    const uint32_t N = A.N[pix];
    if (WHAT == AMAP_SAMPLES) {
        static_cast<uint32_t*>(out)[ob] = N;
        return;
    }
    float* o = static_cast<float*>(out) + 3 * ob;
    for (int ch = 0; ch < 3; ++ch) {
        if (WHAT == AMAP_IMAGE) {
            o[ch] = (float)__ddiv_rn(A.S[3 * pix + ch], (double)N);
        } else {
            const uint32_t K = A.K[pix];
            o[ch] = K < 2 ? __int_as_float(0x7f800000) : (float)__dsqrt_rn(adaptive_e2(A.S[3 * pix + ch], A.Q[3 * pix + ch], N, K));
        }
    }
}

__global__ void k_iota(uint32_t* __restrict__ out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = i;
}

// output stage: gamma_correction (image.rs:53-57) + to_rgb8 (clamp, x255, round) — §8(f) N2
__global__ void k_encode_rgb8(const float* __restrict__ rgb, size_t n, float gamma, uint8_t* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v = powf(rgb[i], gamma);
    v = fminf(fmaxf(v, 0.0f), 1.0f);       // f32::clamp; NaN stays NaN and casts to 0 like NumCast would reject -> 0
    float q = roundf(v * 255.0f);          // f32::round: half away from zero
    out[i] = (v == v) ? (uint8_t)q : (uint8_t)0;
}

// ------------------------------------------------------------------ fused persistent kernel
// The persistent traverse loop of k_wf_extend, but a lane whose ray is finished does not write a hit record and
// fetch somebody else's ray: it waits until at least NRRT_FUSED_MIN lanes of its warp are in the same position,
// then those lanes shade, scatter (or regenerate the next sample / fetch the next work item) and start traversing
// their own next ray, all together.  Path state lives in shared memory (ray, throughput, running sum, hit
// attributes, object-space ray, time: 27 doubles per thread), so neither rays nor hit records ever round-trip
// through HBM and there is no queue, no compaction and a single launch.  Traversal and shading use the same device functions as the
// wavefront kernels and the same (pixel, sample-chunk) work items, so the image is bit-identical.
#ifndef NRRT_FUSED_MIN
#define NRRT_FUSED_MIN 24  // lanes of a warp that must be waiting before a shading round runs.  Measured on B200, round 2
                           // (Cornell / spheres / noise / earth, Mrays/s; profiles/r02_fused_quorum_sweep.log): 16 6173 / 4558 /
                           // 5009 / 10745, 20 6250 / 4645 / 5334 / -, 24 6251 / 4671 / 5539 / 11622, 28 6053 / 4646 / 5596 /
                           // 11929, 32 5486 / 4405 / 5651 / 11875.  (The mesh scenes, which preferred 16-20 in this kernel,
                           // are rendered by the pooled kernel under NRRT_MODE_AUTO.)
#endif
#define NRRT_FUSED_STATE_DOUBLES 27  // o(3) d(3) T(3) sum(3) | attr: p(3) alpha beta dobj(3) | object-space ray (6) | time
#ifndef NRRT_FUSED_BLOCKS_PER_SM
#define NRRT_FUSED_BLOCKS_PER_SM 4   // resident blocks the kernel is compiled for (measured: 4 beats 3 on every scene)
#endif
#define NRRT_FUSED_TRIVIAL_MAX 8      // queries finished inside begin() that a lane absorbs per shading round
#define NRRT_FUSED_STATE_WORDS 4     // item, pixel x, pixel y, sample_end (touched only between paths)
struct SmemCtx {
    static constexpr bool kRayInCtx = true;
    double* st;  // this thread's column: st[k * NRRT_BLOCK]
    __device__ __forceinline__ double time() const { return st[26 * NRRT_BLOCK]; }
    __device__ __forceinline__ void get_obj(d3& oo, d3& dd) const {
        oo = mk3(st[20 * NRRT_BLOCK], st[21 * NRRT_BLOCK], st[22 * NRRT_BLOCK]);
        dd = mk3(st[23 * NRRT_BLOCK], st[24 * NRRT_BLOCK], st[25 * NRRT_BLOCK]);
    }
    __device__ __forceinline__ void put_obj(d3 oo, d3 dd) const {
        st[20 * NRRT_BLOCK] = oo.x, st[21 * NRRT_BLOCK] = oo.y, st[22 * NRRT_BLOCK] = oo.z;
        st[23 * NRRT_BLOCK] = dd.x, st[24 * NRRT_BLOCK] = dd.y, st[25 * NRRT_BLOCK] = dd.z;
    }
    __device__ __forceinline__ void get(d3& oo, d3& dd) const {
        oo = mk3(st[0], st[NRRT_BLOCK], st[2 * NRRT_BLOCK]);
        dd = mk3(st[3 * NRRT_BLOCK], st[4 * NRRT_BLOCK], st[5 * NRRT_BLOCK]);
    }
    __device__ __forceinline__ void put(uint32_t level, d3 p, double a, double b, d3 dobj) const {
        st[12 * NRRT_BLOCK] = p.x, st[13 * NRRT_BLOCK] = p.y, st[14 * NRRT_BLOCK] = p.z;
        st[15 * NRRT_BLOCK] = a, st[16 * NRRT_BLOCK] = b;
        if (level) st[17 * NRRT_BLOCK] = dobj.x, st[18 * NRRT_BLOCK] = dobj.y, st[19 * NRRT_BLOCK] = dobj.z;
    }
};

// MB = resident blocks per SM the kernel is compiled for (register budget 65536 / (MB * 128)).  Measured on B200
// (Cornell / spheres / teapot, Mseg/s, at the time): 3 blocks 4440 / 2957 / 791, 4 blocks 4770 / 3495 / 940.
// SPEC = speculative traversal (rt_device.cuh), chosen per scene by tree size.
template <uint32_t F, int MB, bool SPEC>
__global__ void __launch_bounds__(NRRT_BLOCK, MB)
k_render_fused(const __grid_constant__ DevScene S, const __grid_constant__ nrrt_camera cam,
               const __grid_constant__ RenderParams P, double* __restrict__ partials,
               unsigned long long* __restrict__ counters) {
    extern __shared__ uint32_t s_mem[];
    uint32_t* stack = s_mem + threadIdx.x;
    double* st = reinterpret_cast<double*>(s_mem + NRRT_STACK_CAP * NRRT_BLOCK) + threadIdx.x;
    const SmemCtx ctx{st};
    // per-path bookkeeping that is only touched between paths lives in shared memory too
    uint32_t* wd = reinterpret_cast<uint32_t*>(reinterpret_cast<double*>(s_mem + NRRT_STACK_CAP * NRRT_BLOCK) +
                                               NRRT_FUSED_STATE_DOUBLES * NRRT_BLOCK) + threadIdx.x;
    uint32_t& s_item = wd[0];
    uint32_t& s_px = wd[NRRT_BLOCK];
    uint32_t& s_py = wd[2 * NRRT_BLOCK];
    uint32_t& s_end = wd[3 * NRRT_BLOCK];
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t segs = 0, paths = 0;  // per-thread; a thread traces far fewer than 2^32 segments

    enum : uint32_t { NEED_ITEM = 0, NEED_PATH = 1, TRAVERSING = 2, HIT_READY = 3, RETIRED = 4 };
    uint32_t state = w < P.n_slots ? NEED_ITEM : RETIRED;  // a partial last block: the surplus threads own no item
    s_item = w;  // the first n_slots items are pre-assigned; the counter starts at n_slots
    s_px = s_py = s_end = 0;
    Sampler smp{P.key, 0u, 0u};
    uint32_t bounce = 0;
    Traversal<false, false, F, SPEC, SPEC> tr;  // deep trees: four-slot nodes + speculation; small ones: binary nodes
    uint32_t wb_next = 0, wb_end = 0;  // this warp's block of work items (warp-uniform)

    for (;;) {
        // ---- shading / regeneration round, voted by the warp
        const unsigned pend = __ballot_sync(0xffffffffu, state != TRAVERSING && state != RETIRED);
        const unsigned trav = __ballot_sync(0xffffffffu, state == TRAVERSING);
        if (pend == 0 && trav == 0) break;
        if (pend && (__popc(pend) >= NRRT_FUSED_MIN || trav == 0)) {
            if (state == HIT_READY) {
                d3 o, d;
                ctx.get(o, d);
                d3 T = mk3(st[6 * NRRT_BLOCK], st[7 * NRRT_BLOCK], st[8 * NRRT_BLOCK]);
                d3 L = mk3(0.0, 0.0, 0.0);
                bool alive;
                const HitId& h = tr.best;
                if (h.prim == NRRT_REF_NONE) {  // camera.rs:298
                    L = mul3(T, ld3(cam.background));
                    alive = false;
                } else {
                    HitRec rec;
                    d3 p_obj = mk3(st[12 * NRRT_BLOCK], st[13 * NRRT_BLOCK], st[14 * NRRT_BLOCK]);
                    d3 d_dir = d;
                    if ((F & NRRT_F_INSTANCES) && h.depth)
                        d_dir = mk3(st[17 * NRRT_BLOCK], st[18 * NRRT_BLOCK], st[19 * NRRT_BLOCK]);
                    double al = 0.0, be = 0.0;
                    if (F & NRRT_F_PLANES) al = st[15 * NRRT_BLOCK], be = st[16 * NRRT_BLOCK];
                    const bool want_uv = (F & NRRT_F_TEXTURED) && (S.material_flags[hit_material<F>(S, h.prim)] & 1u) != 0;
                    resolve_hit_attr<F>(S, h, p_obj, al, be, d_dir, (F & NRRT_F_MOTION) ? ctx.time() : 0.0, want_uv, rec);
                    alive = path_shade<F>(S, cam, rec, smp, o, d, T, L, bounce);
                }
                if (alive) {
                    st[0] = o.x, st[NRRT_BLOCK] = o.y, st[2 * NRRT_BLOCK] = o.z;
                    st[3 * NRRT_BLOCK] = d.x, st[4 * NRRT_BLOCK] = d.y, st[5 * NRRT_BLOCK] = d.z;
                    st[6 * NRRT_BLOCK] = T.x, st[7 * NRRT_BLOCK] = T.y, st[8 * NRRT_BLOCK] = T.z;
                    state = TRAVERSING;
                } else {  // path finished: add it to the item's partial sum (sample order)
                    d3 sum = add3(mk3(st[9 * NRRT_BLOCK], st[10 * NRRT_BLOCK], st[11 * NRRT_BLOCK]), L);
                    ++smp.sample;
                    if (smp.sample >= s_end) {  // item finished: publish, fetch the next one
                        size_t pb = (size_t)s_item * 3;
                        partials[pb] = sum.x, partials[pb + 1] = sum.y, partials[pb + 2] = sum.z;
                        s_item = NRRT_NO_ITEM;  // fetched below, by the warp
                        state = NEED_ITEM;
                    } else {
                        st[9 * NRRT_BLOCK] = sum.x, st[10 * NRRT_BLOCK] = sum.y, st[11 * NRRT_BLOCK] = sum.z;
                        state = NEED_PATH;
                    }
                }
            }
            // Work items come to a WARP in blocks of NRRT_ITEM_BLOCK consecutive ones (= consecutive pixels of one chunk)
            // and its lanes take them from there, so however far the lanes drift apart in time they stay on
            // neighbouring pixels: same materials, same textures, same part of the tree.  One atomic per block.
            {
                const bool want = state == NEED_ITEM && s_item == NRRT_NO_ITEM;
                const unsigned need = __ballot_sync(0xffffffffu, want);
                if (need) {
                    const uint32_t lane = threadIdx.x & 31u, n = __popc(need), rank = __popc(need & ((1u << lane) - 1u));
                    const uint32_t avail = wb_end - wb_next;
                    uint32_t fresh_base = 0, fresh_size = 0;
                    if (n > avail) {
                        const uint32_t leader = __ffs(need) - 1;
                        if (lane == leader) {
                            fresh_size = item_block_size(P, *(volatile unsigned long long*)&counters[5], n - avail);
                            fresh_base = (uint32_t)atomicAdd(&counters[5], (unsigned long long)fresh_size);
                        }
                        fresh_base = __shfl_sync(0xffffffffu, fresh_base, leader);
                        fresh_size = __shfl_sync(0xffffffffu, fresh_size, leader);
                    }
                    if (want) s_item = rank < avail ? wb_next + rank : fresh_base + (rank - avail);
                    if (n > avail) wb_next = fresh_base + (n - avail), wb_end = fresh_base + fresh_size;
                    else wb_next += n;
                }
            }
            if (state == NEED_ITEM) {
                if (s_item >= P.n_items) {
                    state = RETIRED;
                } else {
                    WorkItem wi;
                    smp.sample = decode_item<(F & NRRT_F_ACTIVE) != 0>(cam, P, s_item, wi);
                    smp.pixel = wi.y * cam.width + wi.x;
                    s_px = wi.x, s_py = wi.y, s_end = wi.sample_end;
                    st[9 * NRRT_BLOCK] = 0.0, st[10 * NRRT_BLOCK] = 0.0, st[11 * NRRT_BLOCK] = 0.0;
                    state = NEED_PATH;
                }
            }
            if (state == NEED_PATH) {  // Camera::get_ray for the item's next sample
                d3 o, d;
                double tm;
                camera_ray<(F & NRRT_F_MOTION) != 0>(cam, s_px, s_py, smp, o, d, tm);
                if (F & NRRT_F_MOTION) st[26 * NRRT_BLOCK] = tm;
                st[0] = o.x, st[NRRT_BLOCK] = o.y, st[2 * NRRT_BLOCK] = o.z;
                st[3 * NRRT_BLOCK] = d.x, st[4 * NRRT_BLOCK] = d.y, st[5 * NRRT_BLOCK] = d.z;
                st[6 * NRRT_BLOCK] = 1.0, st[7 * NRRT_BLOCK] = 1.0, st[8 * NRRT_BLOCK] = 1.0;
                bounce = 0;
                ++paths;
                state = TRAVERSING;
            }
            // every lane that just became TRAVERSING starts its query (lanes already traversing keep theirs)
            const bool fresh = (pend >> (threadIdx.x & 31u)) & 1u;
            if (fresh && state == TRAVERSING) {
                tr.begin(S, ctx, 0.001, NRRT_INF, nullptr);
                ++segs;
                // A query that is over the moment it begins (the ray misses the scene's root box — every other camera
                // ray of an object in front of a background) is accounted for on the spot and the lane starts its next
                // sample, instead of spending a traversal round and a shading round on a miss.  Only in the deep-tree
                // instantiations: the extra code costs the small-scene kernels 7-12 % even when it never runs.
                for (int rep = 0; SPEC && tr.cur == NRRT_REF_NONE && rep < NRRT_FUSED_TRIVIAL_MAX; ++rep) {
                    const d3 T = mk3(st[6 * NRRT_BLOCK], st[7 * NRRT_BLOCK], st[8 * NRRT_BLOCK]);
                    const d3 sum = add3(mk3(st[9 * NRRT_BLOCK], st[10 * NRRT_BLOCK], st[11 * NRRT_BLOCK]),
                                        mul3(T, ld3(cam.background)));  // camera.rs:298
                    ++smp.sample;
                    if (smp.sample >= s_end) {  // item finished: publish; the next shading round fetches another
                        size_t pb = (size_t)s_item * 3;
                        partials[pb] = sum.x, partials[pb + 1] = sum.y, partials[pb + 2] = sum.z;
                        s_item = NRRT_NO_ITEM;  // the next shading round fetches one
                        state = NEED_ITEM;
                        break;
                    }
                    st[9 * NRRT_BLOCK] = sum.x, st[10 * NRRT_BLOCK] = sum.y, st[11 * NRRT_BLOCK] = sum.z;
                    d3 o, d;
                    double tm;
                    camera_ray<(F & NRRT_F_MOTION) != 0>(cam, s_px, s_py, smp, o, d, tm);
                    if (F & NRRT_F_MOTION) st[26 * NRRT_BLOCK] = tm;
                    st[0] = o.x, st[NRRT_BLOCK] = o.y, st[2 * NRRT_BLOCK] = o.z;
                    st[3 * NRRT_BLOCK] = d.x, st[4 * NRRT_BLOCK] = d.y, st[5 * NRRT_BLOCK] = d.z;
                    st[6 * NRRT_BLOCK] = 1.0, st[7 * NRRT_BLOCK] = 1.0, st[8 * NRRT_BLOCK] = 1.0;
                    bounce = 0;
                    ++paths;
                    tr.begin(S, ctx, 0.001, NRRT_INF, nullptr);
                    ++segs;
                }
            }
        }
        // ---- one traversal round for the lanes that have a query
        if (tr.round(S, ctx, 0.001, NRRT_INF, stack, NRRT_BLOCK, nullptr, state == TRAVERSING) && state == TRAVERSING)
            state = HIT_READY;
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
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_cnt[0], segs64);
        atomicAdd(&s_cnt[1], paths64);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicAdd(&counters[0], s_cnt[0]);
        atomicAdd(&counters[1], s_cnt[1]);
    }
}

#include "pool_kernel.cuh"

// ------------------------------------------------------------------ wavefront
// SoA path state, one entry per slot (n = n_slots).
struct WfState {
    double* ray;       // [7][n]: ox oy oz dx dy dz time
    double* T;         // [3][n] throughput.  (The radiance of a LIVE path is identically zero: no reference
                       //        material both emits and scatters — material.rs:10-27, diffuse_light.rs — so it
                       //        is not stored; a path contributes T*background or T*emitted when it ends.)
    double* sum;       // [3][n] running partial sum of the slot's current work item
    uint32_t* item;    // [n] current work item
    uint32_t* sample;  // [n] current sample index
    uint32_t* bounce;  // [n]
    double* hit_t;     // [n]
    uint32_t* hit_prim;   // [n]
    uint32_t* hit_inst;   // [MAX_DEPTH][n]: word 0 = depth | inst[0] << 3, words 1.. = inst[1..] (depth >= 2 only)
    double* hit_attr;     // [8][n]: object-space hit point, alpha, beta, object-space direction (MemHitSink)
    uint32_t* queue[2];   // [n] slot indices
    uint32_t* count;      // [2][2] queue lengths: [q][0] = bounce rays, stored at the front of queue q in ascending
                          //        order; [q][1] = freshly generated camera rays, stored from the back in descending
                          //        order.  Camera rays of neighbouring pixels are coherent; keeping them in warps
                          //        of their own (instead of mixing them with incoherent bounce rays) keeps those
                          //        warps converged in the traverse and shade kernels.
    uint32_t* cursor;     // [2] fetch cursors of the persistent extend kernel
    double* partials;     // [n_items][3]
    unsigned long long* counters;  // [0]=segments [1]=paths [5]=next work item
};

// logical queue position i in [0, n_bounce + n_cam) -> physical index in the queue array of n entries
__device__ __forceinline__ uint32_t queue_slot(const uint32_t* q, uint32_t n, uint32_t n_bounce, uint32_t i) {
    return q[i < n_bounce ? i : n - 1u - (i - n_bounce)];
}

// ray generation for the initial items
template <bool ACTIVE>
__global__ void __launch_bounds__(NRRT_BLOCK)
k_wf_init(const __grid_constant__ nrrt_camera cam, const __grid_constant__ RenderParams P,
          const __grid_constant__ WfState W) {
    uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) {
        W.count[0] = NRRT_SPLIT_QUEUE ? 0 : P.n_slots;  // queue 0: no bounce rays yet ...
        W.count[1] = NRRT_SPLIT_QUEUE ? P.n_slots : 0;  // ... every slot starts with a camera ray
        W.count[2] = 0;
        W.count[3] = 0;
        W.cursor[0] = 0;
        W.cursor[1] = 0;
        W.counters[1] += P.n_slots;
    }
    if (w >= P.n_slots) return;
    uint32_t n = P.n_slots;
    WorkItem wi;
    uint32_t first = decode_item<ACTIVE>(cam, P, w, wi);
    Sampler smp{P.key, wi.y * cam.width + wi.x, first};
    d3 o, d;
    double tm;
    camera_ray<true>(cam, wi.x, wi.y, smp, o, d, tm);
    W.ray[6 * (size_t)n + w] = tm;
    W.ray[0 * (size_t)n + w] = o.x, W.ray[1 * (size_t)n + w] = o.y, W.ray[2 * (size_t)n + w] = o.z;
    W.ray[3 * (size_t)n + w] = d.x, W.ray[4 * (size_t)n + w] = d.y, W.ray[5 * (size_t)n + w] = d.z;
    for (int c = 0; c < 3; ++c) {
        W.T[c * (size_t)n + w] = 1.0;
        W.sum[c * (size_t)n + w] = 0.0;
    }
    W.item[w] = w;
    W.sample[w] = first;
    W.bounce[w] = 0;
    W.queue[0][NRRT_SPLIT_QUEUE ? n - 1u - w : w] = w;  // camera-ray region: from the back, descending
}

// traverse / intersect: closest hit for every queued ray.
// Persistent warps with dynamic ray fetch: rays of one warp finish after very different numbers of traversal
// rounds, so lanes whose ray is done pull the next queued ray (warp-aggregated atomicAdd on a cursor) instead of
// idling until the slowest lane of the warp finishes.
#ifndef NRRT_REFILL_MIN
#define NRRT_REFILL_MIN 16  // refill once this many lanes of the warp are idle (8/16 measured: 16 wins on Cornell + teapot)
#endif
#ifndef NRRT_EXTEND_MINBLOCKS
#define NRRT_EXTEND_MINBLOCKS 4  // resident blocks per SM the traverse kernel is compiled for (5 spills since the state moved to registers)
#endif
template <uint32_t F>
__global__ void __launch_bounds__(NRRT_BLOCK, NRRT_EXTEND_MINBLOCKS)
k_wf_extend(const __grid_constant__ DevScene S, const __grid_constant__ WfState W, uint32_t n, uint32_t qin) {
    extern __shared__ uint32_t s_stack[];
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t n_bounce = W.count[2 * qin], n_in = n_bounce + W.count[2 * qin + 1];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        W.count[2 * (qin ^ 1)] = 0;      // the other queue is filled by the next shade pass
        W.count[2 * (qin ^ 1) + 1] = 0;
        W.cursor[qin ^ 1] = 0;           // and consumed by the next extend pass
    }
    Traversal<false, false, F> tr;
    bool has = false, exhausted = false;
    uint32_t slot = 0;
    for (;;) {
        const unsigned idle = __ballot_sync(0xffffffffu, !has);
        if (idle && !exhausted && (idle == 0xffffffffu || __popc(idle) >= NRRT_REFILL_MIN)) {
            const uint32_t want = __popc(idle), leader = __ffs(idle) - 1;
            uint32_t base = 0;
            if (lane == leader) base = atomicAdd(&W.cursor[qin], want);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + want >= n_in) exhausted = true;
            if (!has) {
                uint32_t i = base + __popc(idle & ((1u << lane) - 1u));
                if (i < n_in) {
                    slot = queue_slot(W.queue[qin], n, n_bounce, i);
                    tr.begin(S, MemCtx{W.ray, W.hit_attr, n, slot}, 0.001, NRRT_INF, nullptr);
                    has = true;
                }
            }
        }
        if (__ballot_sync(0xffffffffu, has) == 0) break;
        if (tr.round(S, MemCtx{W.ray, W.hit_attr, n, slot}, 0.001, NRRT_INF, s_stack + threadIdx.x, NRRT_BLOCK, nullptr,
                     has) && has) {
            W.hit_t[slot] = tr.best.t;
            W.hit_prim[slot] = tr.best.prim;
            if (F & NRRT_F_INSTANCES) W.hit_inst[slot] = tr.best.depth | (tr.best.inst.a << 3);
            if ((F & NRRT_F_INSTANCES) && tr.best.depth > 1)
                for (uint32_t l = 1; l < tr.best.depth; ++l) W.hit_inst[(size_t)l * n + slot] = tr.best.inst.get(l);
            has = false;
        }
    }
}

// shade / scatter, in-slot path regeneration, dynamic work fetch, warp-ballot compaction of the survivors
#ifndef NRRT_SHADE_MINBLOCKS
#define NRRT_SHADE_MINBLOCKS 6
#endif
template <uint32_t F>
__global__ void __launch_bounds__(NRRT_BLOCK, NRRT_SHADE_MINBLOCKS)
k_wf_shade(const __grid_constant__ DevScene S, const __grid_constant__ nrrt_camera cam,
           const __grid_constant__ RenderParams P, const __grid_constant__ WfState W, uint32_t qin) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n = P.n_slots;
    const uint32_t n_bounce = W.count[2 * qin], n_in = n_bounce + W.count[2 * qin + 1];
    const uint32_t lane_id = threadIdx.x & 31u;
    if (i == 0) W.counters[0] += n_in;  // one closest-hit query per queued ray
    bool active = i < n_in, survive = false, need_item = false, new_path = false;
    uint32_t slot = 0, item = 0, bounce = 0;
    d3 o, d, T, L, sum;
    Sampler smp{P.key, 0u, 0u};
    WorkItem wi;
    if (active) {
        slot = queue_slot(W.queue[qin], n, n_bounce, i);
        o = mk3(W.ray[slot], W.ray[(size_t)n + slot], W.ray[2 * (size_t)n + slot]);
        d = mk3(W.ray[3 * (size_t)n + slot], W.ray[4 * (size_t)n + slot], W.ray[5 * (size_t)n + slot]);
        T = mk3(W.T[slot], W.T[(size_t)n + slot], W.T[2 * (size_t)n + slot]);
        L = mk3(0.0, 0.0, 0.0);
        bounce = W.bounce[slot];
        item = W.item[slot];
        decode_item<(F & NRRT_F_ACTIVE) != 0>(cam, P, item, wi);
        smp.pixel = wi.y * cam.width + wi.x;
        smp.sample = W.sample[slot];
        HitId h;
        h.t = W.hit_t[slot];
        h.prim = W.hit_prim[slot];
        {
            const uint32_t w0 = (!(F & NRRT_F_INSTANCES) || h.prim == NRRT_REF_NONE) ? 0u : W.hit_inst[slot];
            h.depth = w0 & 7u;
            h.inst.clear();
            h.inst.a = w0 >> 3;
#pragma unroll
            for (uint32_t l = 1; l < NRRT_MAX_INSTANCE_DEPTH; ++l)
                h.inst.set(l, ((F & NRRT_F_INSTANCES) && l < h.depth) ? W.hit_inst[(size_t)l * n + slot] : 0u);
        }
#if !NRRT_HIT_SINK
        survive = path_step(S, cam, h, smp, o, d, W.ray[6 * (size_t)n + slot], T, L, bounce);
#else
        if (h.prim == NRRT_REF_NONE) {  // camera.rs:298
            L = mul3(T, ld3(cam.background));
            survive = false;
        } else {
            HitRec rec;
            const double* A = W.hit_attr;
            d3 p_obj = mk3(A[slot], A[(size_t)n + slot], A[2 * (size_t)n + slot]);
            d3 d_dir = d;
            if ((F & NRRT_F_INSTANCES) && h.depth)
                d_dir = mk3(A[5 * (size_t)n + slot], A[6 * (size_t)n + slot], A[7 * (size_t)n + slot]);
            double al = 0.0, be = 0.0;
            if (F & NRRT_F_PLANES) al = A[3 * (size_t)n + slot], be = A[4 * (size_t)n + slot];
            const bool want_uv = (F & NRRT_F_TEXTURED) && (S.material_flags[hit_material<F>(S, h.prim)] & 1u) != 0;
            resolve_hit_attr<F>(S, h, p_obj, al, be, d_dir, (F & NRRT_F_MOTION) ? W.ray[6 * (size_t)n + slot] : 0.0, want_uv,
                                rec);
            survive = path_shade<F>(S, cam, rec, smp, o, d, T, L, bounce);
        }
#endif
        if (!survive) {  // path finished: add it to the item's partial sum (sample order)
            sum = add3(mk3(W.sum[slot], W.sum[(size_t)n + slot], W.sum[2 * (size_t)n + slot]), L);
            ++smp.sample;
            if (smp.sample >= wi.sample_end) {  // item finished: publish, then fetch another below
                size_t pb = (size_t)item * 3;
                W.partials[pb] = sum.x, W.partials[pb + 1] = sum.y, W.partials[pb + 2] = sum.z;
                sum = mk3(0.0, 0.0, 0.0);
                need_item = true;
            } else {
                new_path = true;
            }
        }
    }
    // warp-aggregated fetch from the global work counter
    unsigned need = __ballot_sync(0xffffffffu, need_item);
    if (need) {
        uint32_t leader = __ffs(need) - 1, base = 0;
        if (lane_id == leader) base = (uint32_t)atomicAdd(&W.counters[5], (unsigned long long)__popc(need));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (need_item) {
            item = base + __popc(need & ((1u << lane_id) - 1u));
            if (item < P.n_items) {
                smp.sample = decode_item<(F & NRRT_F_ACTIVE) != 0>(cam, P, item, wi);
                smp.pixel = wi.y * cam.width + wi.x;
                W.item[slot] = item;
                new_path = true;
            }
        }
    }
    if (active && !survive) {
        W.sum[slot] = sum.x, W.sum[(size_t)n + slot] = sum.y, W.sum[2 * (size_t)n + slot] = sum.z;
        if (new_path) {  // regenerate in place: next sample of the item
            double tm;
            camera_ray<(F & NRRT_F_MOTION) != 0>(cam, wi.x, wi.y, smp, o, d, tm);
            if (F & NRRT_F_MOTION) W.ray[6 * (size_t)n + slot] = tm;
            T = mk3(1.0, 1.0, 1.0);
            L = mk3(0.0, 0.0, 0.0);
            bounce = 0;
            survive = true;
            W.sample[slot] = smp.sample;
        }
    }
    unsigned born = __ballot_sync(0xffffffffu, new_path);
    if (born && lane_id == 0) atomicAdd(&W.counters[1], (unsigned long long)__popc(born));
    if (survive) {
        W.ray[slot] = o.x, W.ray[(size_t)n + slot] = o.y, W.ray[2 * (size_t)n + slot] = o.z;
        W.ray[3 * (size_t)n + slot] = d.x, W.ray[4 * (size_t)n + slot] = d.y, W.ray[5 * (size_t)n + slot] = d.z;
        W.T[slot] = T.x, W.T[(size_t)n + slot] = T.y, W.T[2 * (size_t)n + slot] = T.z;
        W.bounce[slot] = bounce;
    }
    // warp-aggregated compaction of the survivors into the other queue: bounce rays to the front, freshly generated
    // camera rays to the back
    const bool cam_ray = NRRT_SPLIT_QUEUE && survive && new_path;
    const unsigned b_bounce = __ballot_sync(0xffffffffu, survive && !cam_ray), b_cam = __ballot_sync(0xffffffffu, cam_ray);
    if (b_bounce | b_cam) {
        uint32_t base_b = 0, base_c = 0;
        if (lane_id == 0) {
            if (b_bounce) base_b = atomicAdd(&W.count[2 * (qin ^ 1)], (uint32_t)__popc(b_bounce));
            if (b_cam) base_c = atomicAdd(&W.count[2 * (qin ^ 1) + 1], (uint32_t)__popc(b_cam));
        }
        base_b = __shfl_sync(0xffffffffu, base_b, 0);
        base_c = __shfl_sync(0xffffffffu, base_c, 0);
        const unsigned below = (1u << lane_id) - 1u;
        if (survive && !cam_ray) W.queue[qin ^ 1][base_b + __popc(b_bounce & below)] = slot;
        if (cam_ray) W.queue[qin ^ 1][n - 1u - (base_c + __popc(b_cam & below))] = slot;
    }
}

// =========================================================================== host side of the ABI
static thread_local std::string g_create_error;  // per thread: nrrt_create may run on several threads (nrrt_render_multi)

struct nrrt_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    bool has_scene = false;
    DevScene dev{};
    uint32_t max_stack = 0;
    std::vector<void*> scene_allocs;
    std::vector<cudaTextureObject_t> tex_objs;
    std::vector<cudaArray_t> tex_arrays;
    // scratch
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    unsigned long long* d_counters = nullptr;  // 8 x u64
    uint32_t* h_count = nullptr;               // pinned, polling ring
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> ev_pool;
    unsigned persistent_blocks = 592;  // SMs x resident blocks of the extend kernel
    unsigned sms = 148;                // multiprocessors
    size_t smem_per_sm = 228 * 1024, smem_per_block = 227 * 1024;  // shared memory limits (opt-in)
    uint32_t features = NRRT_F_ALL;    // NRRT_F_* mask of the uploaded scene
    double trace_time = 0.0;           // Ray::time of nrrt_trace_rays queries
    bool speculate = false;            // fused kernel: speculative traversal (deep trees only)
    bool has_binary = false;           // the scene also went up in binary-node form (small trees)
    uint32_t binary_stack = 0;         // traversal stack need over the binary nodes
    cudaStream_t side = nullptr;       // progress polling while a single-launch render runs (created on first use)
    void* enc_buf = nullptr;           // output-stage scratch (nrrt_encode_rgb8), grown on demand
    size_t enc_bytes = 0;
    uint64_t scene_gen = 0;            // bumped by every nrrt_scene_upload: an nrrt_accum belongs to one scene
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
            return NRRT_ERR_CUDA;                                                                  \
        }                                                                                          \
    } while (0)

static void free_scene(nrrt_ctx* ctx) {
    for (auto t : ctx->tex_objs) cudaDestroyTextureObject(t);
    for (auto a : ctx->tex_arrays) cudaFreeArray(a);
    for (void* p : ctx->scene_allocs) cudaFree(p);
    ctx->tex_objs.clear();
    ctx->tex_arrays.clear();
    ctx->scene_allocs.clear();
    ctx->has_scene = false;
}

template <class T>
static int upload(nrrt_ctx* ctx, const T* host, size_t count, const T** dev_out) {
    *dev_out = nullptr;
    size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
    void* p = nullptr;
    CK(cudaMalloc(&p, bytes));
    ctx->scene_allocs.push_back(p);
    if (count) {
        if (!host) {
            ctx->err = "scene array pointer is NULL";
            return NRRT_ERR_INVALID;
        }
        CK(cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    }
    *dev_out = (const T*)p;
    return NRRT_OK;
}

// noise 0.9.0 PermutationTable::new(seed): XorShiftRng seeded with [1, s, s, s] driving rand 0.8.5's
// Fisher-Yates shuffle of 0..255 (SURVEY.md note A; recalled from the published sources, unpinned).
static void noise_perm_table(uint32_t seed, uint8_t* out) {
    uint32_t x = 1, y = seed, z = seed, w = seed;
    for (int i = 0; i < 256; ++i) out[i] = (uint8_t)i;
    for (uint32_t i = 255; i >= 1; --i) {
        uint32_t range = i + 1, zone = (range << __builtin_clz(range)) - 1u, pick;
        for (;;) {
            uint32_t t = x ^ (x << 11);
            x = y, y = z, z = w;
            w = w ^ (w >> 19) ^ (t ^ (t >> 8));
            uint64_t m = (uint64_t)w * range;
            if ((uint32_t)m <= zone) {
                pick = (uint32_t)(m >> 32);
                break;
            }
        }
        std::swap(out[i], out[pick]);
    }
}

extern "C" {

int nrrt_create(int device, nrrt_ctx** out) {
    if (!out) return NRRT_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) +
                         "); this library has no CPU fallback";
        return NRRT_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) {
        g_create_error = "device index out of range";
        return NRRT_ERR_INVALID;
    }
    nrrt_ctx* ctx = new nrrt_ctx();
    ctx->device = device;
    auto bail = [&](const char* what, cudaError_t err) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
        delete ctx;
        return NRRT_ERR_CUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) {
            ctx->persistent_blocks = (unsigned)sms * NRRT_EXTEND_MINBLOCKS;
            ctx->sms = (unsigned)sms;
        }
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device) == cudaSuccess && v > 0)
            ctx->smem_per_sm = (size_t)v;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) == cudaSuccess && v > 0)
            ctx->smem_per_block = (size_t)v;
    }
    if ((e = cudaMalloc((void**)&ctx->d_counters, 8 * sizeof(unsigned long long))) != cudaSuccess)
        return bail("cudaMalloc", e);
    if ((e = cudaMallocHost((void**)&ctx->h_count, 128 * sizeof(uint32_t))) != cudaSuccess)
        return bail("cudaMallocHost", e);
    if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return bail("cudaEventCreate", e);
    *out = ctx;
    return NRRT_OK;
}

void nrrt_destroy(nrrt_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    free_scene(ctx);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->enc_buf) cudaFree(ctx->enc_buf);
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    if (ctx->h_count) cudaFreeHost(ctx->h_count);
    if (ctx->side) cudaStreamDestroy(ctx->side);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    delete ctx;
}

const char* nrrt_last_error(const nrrt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int nrrt_set_stream(nrrt_ctx* ctx, void* cuda_stream) {
    if (!ctx) return NRRT_ERR_INVALID;
    ctx->stream = (cudaStream_t)cuda_stream;
    return NRRT_OK;
}

int nrrt_set_trace_time(nrrt_ctx* ctx, double time) {
    if (!ctx) return NRRT_ERR_INVALID;
    ctx->trace_time = time;
    return NRRT_OK;
}

static uint32_t pick_features(uint32_t need);
#define NRRT_BINARY_MAX_NODES 64u  // scenes with fewer inner nodes are also uploaded in binary form (fused kernel)
#define NRRT_POOL_MIN_NODES 1024u  // NRRT_MODE_AUTO: four-slot nodes from which the pooled kernel is the product path

// Stack entries a traversal of the binary nodes can need, or a value above any cap when the arrays are unusable
// (a reference out of range, children not after their parents).  Same sweep as for the four-slot nodes.
static uint32_t binary_stack_need(const nrrt_scene_desc* sc) {
    const uint32_t bad = 1u << 20;
    if (!sc->nodes || !sc->child_boxes) return bad;
    auto ok = [&](uint32_t r) {
        if (r == NRRT_REF_NONE) return true;
        const uint32_t ix = NRRT_REF_INDEX(r);
        switch (NRRT_REF_TYPE(r)) {
            case NRRT_REF_NODE: return ix < sc->n_nodes;
            case NRRT_REF_SPHERE: return ix < sc->n_spheres;
            case NRRT_REF_PLANE: return ix < sc->n_planes;
            case NRRT_REF_INSTANCE: return ix < sc->n_instances;
            default: return false;
        }
    };
    if (!ok(sc->root)) return bad;
    for (uint32_t i = 0; i < sc->n_instances; ++i)
        if (!ok(sc->instances[i].inner)) return bad;
    for (uint32_t i = 0; i < sc->n_nodes; ++i)
        for (int c = 0; c < 2; ++c) {
            const uint32_t r = sc->nodes[i].child[c];
            if (!ok(r)) return bad;
            if (r != NRRT_REF_NONE && NRRT_REF_TYPE(r) == NRRT_REF_NODE && NRRT_REF_INDEX(r) <= i) return bad;
        }
    std::vector<uint32_t> need(sc->n_nodes, 0), inst_need(sc->n_instances, 1);
    auto below = [&](uint32_t r) -> uint32_t {
        if (r == NRRT_REF_NONE) return 0;
        if (NRRT_REF_TYPE(r) == NRRT_REF_NODE) return need[NRRT_REF_INDEX(r)];
        if (NRRT_REF_TYPE(r) == NRRT_REF_INSTANCE) return inst_need[NRRT_REF_INDEX(r)];
        return 0;
    };
    for (int sweep = 0;; ++sweep) {
        bool changed = false;
        for (uint32_t i = sc->n_nodes; i-- > 0;) {
            const uint32_t v = std::max(below(sc->nodes[i].child[0]), below(sc->nodes[i].child[1])) + 1;
            if (v != need[i]) need[i] = v, changed = true;
        }
        for (uint32_t i = 0; i < sc->n_instances; ++i) {
            const uint32_t v = below(sc->instances[i].inner) + 1;
            if (v != inst_need[i]) inst_need[i] = v, changed = true;
        }
        if (!changed) break;
        if (sweep > NRRT_MAX_INSTANCE_DEPTH + 1) return bad;
    }
    return below(sc->root);
}

// The flat scene is plain caller memory: check every reference and index the kernels will follow, and recompute the
// traversal stack need instead of trusting max_stack, so a stale or corrupted description is refused here rather than
// overrunning a thread's shared-memory stack or reading out of bounds on the device.  Returns "" when sound.
static std::string validate_scene_desc(const nrrt_scene_desc* sc) {
    auto need_ptr = [](const void* p, uint64_t n) { return n == 0 || p != nullptr; };
    if (!need_ptr(sc->wnodes, sc->n_wnodes) || !need_ptr(sc->wide_boxes, sc->n_wnodes)) return "wide node arrays missing";
    if (!need_ptr(sc->sphere_rec, sc->n_spheres) || !need_ptr(sc->sphere_material, sc->n_spheres) ||
        !need_ptr(sc->sphere_order, sc->n_spheres) || !need_ptr(sc->sphere_object, sc->n_spheres))
        return "sphere arrays missing";
    if (!need_ptr(sc->plane_rec, sc->n_planes) || !need_ptr(sc->plane_material, sc->n_planes) ||
        !need_ptr(sc->plane_order, sc->n_planes) || !need_ptr(sc->plane_object, sc->n_planes))
        return "plane arrays missing";
    if (!need_ptr(sc->instances, sc->n_instances) || !need_ptr(sc->instance_order, sc->n_instances) ||
        !need_ptr(sc->instance_wide_inner, sc->n_instances) || !need_ptr(sc->xforms, sc->n_xforms))
        return "instance arrays missing";
    if (!need_ptr(sc->materials, sc->n_materials) || !need_ptr(sc->textures, sc->n_textures) ||
        !need_ptr(sc->images, sc->n_images))
        return "shading tables missing";
    auto ref_ok = [&](uint32_t r) {
        if (r == NRRT_REF_NONE) return true;
        const uint32_t ix = NRRT_REF_INDEX(r);
        switch (NRRT_REF_TYPE(r)) {
            case NRRT_REF_NODE: return ix < sc->n_wnodes;
            case NRRT_REF_SPHERE: return ix < sc->n_spheres;
            case NRRT_REF_PLANE: return ix < sc->n_planes;
            case NRRT_REF_INSTANCE: return ix < sc->n_instances;
            default: return false;
        }
    };
    if (!ref_ok(sc->wide_root)) return "root reference out of range";
    for (uint32_t i = 0; i < sc->n_wnodes; ++i)
        for (int s = 0; s < 4; ++s) {
            const uint32_t r = sc->wnodes[i].child[s];
            if (!ref_ok(r)) return "node child reference out of range";
            if (r != NRRT_REF_NONE && NRRT_REF_TYPE(r) == NRRT_REF_NODE && NRRT_REF_INDEX(r) <= i)
                return "node children must follow their parent (depth-first order)";  // also rules out cycles
        }
    for (uint32_t i = 0; i < sc->n_instances; ++i) {
        const nrrt_instance& in = sc->instances[i];
        if (!ref_ok(sc->instance_wide_inner[i])) return "instance inner reference out of range";
        if ((uint64_t)in.first_xform + in.n_xforms > sc->n_xforms) return "instance transform range out of bounds";
    }
    for (uint32_t i = 0; i < sc->n_xforms; ++i)
        if (sc->xforms[i].kind > NRRT_XF_SCALE) return "unknown transform kind";
    for (uint32_t i = 0; i < sc->n_spheres; ++i)
        if (sc->sphere_material[i] >= sc->n_materials) return "sphere material out of range";
    for (uint32_t i = 0; i < sc->n_planes; ++i)
        if ((sc->plane_material[i] & ~NRRT_PLANE_TRIANGLE_BIT) >= sc->n_materials) return "plane material out of range";
    for (uint32_t i = 0; i < sc->n_materials; ++i) {
        const nrrt_material& m = sc->materials[i];
        if (m.kind > NRRT_MAT_DIFFUSE_LIGHT) return "unknown material kind";
        if (m.kind != NRRT_MAT_DIELECTRIC && m.texture >= sc->n_textures) return "material texture out of range";
    }
    for (uint32_t i = 0; i < sc->n_textures; ++i) {
        const nrrt_texture& t = sc->textures[i];
        if (t.kind > NRRT_TEX_MARBLE) return "unknown texture kind";
        if (t.kind == NRRT_TEX_CHECKER && (t.a >= i || t.b >= i)) return "checker sub-textures must precede the checker";
        if (t.kind == NRRT_TEX_IMAGE && t.a >= sc->n_images) return "image index out of range";
    }
    // worst-case stack need: node -> node edges only go to larger indices, so one reverse sweep settles a space;
    // instances reach into other spaces (possibly emitted earlier), so sweep until nothing changes — one sweep per
    // nesting level; still changing after NRRT_MAX_INSTANCE_DEPTH + 1 sweeps means too deep a nesting or a cycle
    std::vector<uint32_t> need(sc->n_wnodes, 0), inst_need(sc->n_instances, 1);
    auto below = [&](uint32_t r) -> uint32_t {
        if (r == NRRT_REF_NONE) return 0;
        if (NRRT_REF_TYPE(r) == NRRT_REF_NODE) return need[NRRT_REF_INDEX(r)];
        if (NRRT_REF_TYPE(r) == NRRT_REF_INSTANCE) return inst_need[NRRT_REF_INDEX(r)];
        return 0;
    };
    for (int sweep = 0;; ++sweep) {
        bool changed = false;
        for (uint32_t i = sc->n_wnodes; i-- > 0;) {
            uint32_t deepest = 0, n = 0;
            for (int s = 0; s < 4; ++s) {
                const uint32_t r = sc->wnodes[i].child[s];
                if (r == NRRT_REF_NONE) continue;
                ++n;
                deepest = std::max(deepest, below(r));
            }
            const uint32_t v = deepest + (n ? n - 1 : 0);
            if (v != need[i]) need[i] = v, changed = true;
        }
        for (uint32_t i = 0; i < sc->n_instances; ++i) {
            const uint32_t v = below(sc->instance_wide_inner[i]) + 1;  // the level marker
            if (v != inst_need[i]) inst_need[i] = v, changed = true;
        }
        if (!changed) break;
        if (sweep > NRRT_MAX_INSTANCE_DEPTH + 1) return "instances nest deeper than NRRT_MAX_INSTANCE_DEPTH (or form a cycle)";
    }
    const uint32_t total = below(sc->wide_root);
    if (total + 2 > NRRT_STACK_CAP) return "scene needs a deeper traversal stack than NRRT_STACK_CAP";
    return "";
}

int nrrt_scene_upload(nrrt_ctx* ctx, const nrrt_scene_desc* sc) {
    if (!ctx || !sc) return NRRT_ERR_INVALID;
    if (sc->abi_version != NRRT_ABI_VERSION) {
        ctx->err = "scene desc ABI version mismatch";
        return NRRT_ERR_INVALID;
    }
    {
        std::string why = validate_scene_desc(sc);
        if (!why.empty()) {
            ctx->err = "nrrt_scene_upload: " + why;
            return why.find("stack") != std::string::npos ? NRRT_ERR_LIMIT : NRRT_ERR_INVALID;
        }
    }
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    free_scene(ctx);
    ++ctx->scene_gen;
    DevScene D{};
    int rc;
#define UP(field, host, count)                                          \
    if ((rc = upload(ctx, host, count, &D.field)) != NRRT_OK) {         \
        free_scene(ctx);                                                \
        return rc;                                                      \
    }
    const float4* wnodes4 = nullptr;
    if ((rc = upload(ctx, (const float4*)sc->wnodes, (size_t)sc->n_wnodes * 8, &wnodes4)) != NRRT_OK) {
        free_scene(ctx);
        return rc;
    }
    D.wnodes = wnodes4;
    UP(wide_boxes, sc->wide_boxes, (size_t)sc->n_wnodes * 8);
    D.root = sc->wide_root;
    D.root_box = sc->root_box;
    // small trees also go up in binary form (see DevScene::bnodes); validate_scene_desc checked them
    const bool binary_ok = sc->nodes && sc->child_boxes && sc->n_nodes > 0 && sc->n_nodes < NRRT_BINARY_MAX_NODES &&
                           binary_stack_need(sc) + 2 <= NRRT_STACK_CAP;
    if (binary_ok) {
        const float4* bn = nullptr;
        if ((rc = upload(ctx, (const float4*)sc->nodes, (size_t)sc->n_nodes * 4, &bn)) != NRRT_OK) {
            free_scene(ctx);
            return rc;
        }
        D.bnodes = bn;
        UP(bchild_boxes, sc->child_boxes, (size_t)sc->n_nodes * 2);
        std::vector<uint32_t> binner(std::max<uint32_t>(sc->n_instances, 1), NRRT_REF_NONE);
        for (uint32_t i = 0; i < sc->n_instances; ++i) binner[i] = sc->instances[i].inner;
        UP(inst_binner, binner.data(), binner.size());
        D.broot = sc->root;
    }
    UP(sphere_rec, sc->sphere_rec, (size_t)sc->n_spheres * 4);
    if (sc->n_spheres && sc->sphere_speed) {
        UP(sphere_speed, sc->sphere_speed, (size_t)sc->n_spheres * 3);
    } else {
        D.sphere_speed = nullptr;
    }
    UP(sphere_material, sc->sphere_material, sc->n_spheres);
    UP(sphere_order, sc->sphere_order, sc->n_spheres);
    UP(sphere_object, sc->sphere_object, sc->n_spheres);
    UP(plane_rec, sc->plane_rec, (size_t)sc->n_planes * 16);
    {   // f32 reject-only records (plane_prereject): A = v x w, B = w x u in f64, then rounded
        std::vector<float4> p32((size_t)sc->n_planes * 4);
        for (uint32_t i = 0; i < sc->n_planes; ++i) {
            const double* r = sc->plane_rec + 16 * (size_t)i;  // normal, d, p, w, u, v
            const double *n = r, *pp = r + 4, *w = r + 7, *u = r + 10, *v = r + 13;
            const double A[3] = {v[1] * w[2] - v[2] * w[1], v[2] * w[0] - v[0] * w[2], v[0] * w[1] - v[1] * w[0]};
            const double B[3] = {w[1] * u[2] - w[2] * u[1], w[2] * u[0] - w[0] * u[2], w[0] * u[1] - w[1] * u[0]};
            // |A|_1, |B|_1, |p|_inf rounded UP (they scale error bounds)
            auto up = [](double x) { float f = (float)x; return (double)f < x ? std::nextafterf(f, INFINITY) : f; };
            float a1 = up(std::fabs(A[0]) + std::fabs(A[1]) + std::fabs(A[2])) * 1.0000002f;
            const float b1 = up(std::fabs(B[0]) + std::fabs(B[1]) + std::fabs(B[2])) * 1.0000002f;
            const float pmax = up(std::fmax(std::fmax(std::fabs(pp[0]), std::fabs(pp[1])), std::fabs(pp[2])));
            if (sc->plane_material[i] & NRRT_PLANE_TRIANGLE_BIT) a1 = -a1;  // sign bit = Triangle (NaN keeps "maybe")
            p32[4 * (size_t)i + 0] = make_float4((float)n[0], (float)n[1], (float)n[2], (float)r[3]);
            p32[4 * (size_t)i + 1] = make_float4((float)A[0], (float)A[1], (float)A[2], (float)pp[0]);
            p32[4 * (size_t)i + 2] = make_float4((float)B[0], (float)B[1], (float)B[2], (float)pp[1]);
            p32[4 * (size_t)i + 3] = make_float4((float)pp[2], a1, b1, pmax);
        }
        UP(plane32, p32.data(), p32.size());
    }
    UP(plane_material, sc->plane_material, sc->n_planes);
    UP(plane_order, sc->plane_order, sc->n_planes);
    UP(plane_object, sc->plane_object, sc->n_planes);
    std::vector<nrrt_instance> inst(sc->instances, sc->instances + sc->n_instances);
    for (uint32_t i = 0; i < sc->n_instances; ++i) inst[i].inner = sc->instance_wide_inner[i];  // the kernels walk wide nodes
    UP(instances, inst.data(), inst.size());
    UP(instance_order, sc->instance_order, sc->n_instances);
    UP(xforms, sc->xforms, sc->n_xforms);
    UP(materials, sc->materials, sc->n_materials);

    // textures: fill noise defaults + the Fbm scale factor, build permutation tables
    std::vector<nrrt_texture> tex(sc->textures, sc->textures + sc->n_textures);
    std::vector<uint32_t> perm_base(std::max<uint32_t>(sc->n_textures, 1), 0);
    std::vector<uint8_t> perm;
    for (uint32_t i = 0; i < sc->n_textures; ++i) {
        nrrt_texture& t = tex[i];
        if (t.kind == NRRT_TEX_MARBLE) {  // Fbm::new(seed).set_octaves(7).set_frequency(f)  marble.rs:50-54
            t.octaves = 7;
            t.f1 = 3.14159265358979323846264338327950288 * 2.0 / 3.0;
            t.f2 = 0.5;
        }
        if (t.kind == NRRT_TEX_NOISE || t.kind == NRRT_TEX_MARBLE) {
            t.octaves = std::min<uint32_t>(std::max<uint32_t>(t.octaves, 1u), 32u);
            double denom = 0.0;
            for (uint32_t k = 1; k <= t.octaves; ++k) {  // 1 / sum persistence^k (powi by squaring)
                double pw = 1.0, base = t.f2;
                for (uint32_t e = k;;) {
                    if (e & 1u) pw *= base;
                    e >>= 1;
                    if (!e) break;
                    base *= base;
                }
                denom = denom + pw;
            }
            t.color[0] = 1.0 / denom;
            perm_base[i] = (uint32_t)(perm.size() / 256);
            for (uint32_t k = 0; k < t.octaves; ++k) {
                perm.resize(perm.size() + 256);
                noise_perm_table(t.seed + k, perm.data() + perm.size() - 256);
            }
        }
    }
    UP(textures, tex.data(), tex.size());
    UP(perm, perm.data(), perm.size());
    UP(perm_base, perm_base.data(), perm_base.size());

    // per-material flag: does the texture chain read uv?  (checker.rs:82, image.rs:36-37)
    std::vector<uint8_t> mflags(std::max<uint32_t>(sc->n_materials, 1), 0);
    for (uint32_t i = 0; i < sc->n_materials; ++i) {
        if (sc->materials[i].kind == NRRT_MAT_DIELECTRIC) continue;
        uint32_t ti = sc->materials[i].texture;
        if (ti < sc->n_textures && (tex[ti].kind == NRRT_TEX_CHECKER || tex[ti].kind == NRRT_TEX_IMAGE)) mflags[i] = 1;
    }
    UP(material_flags, mflags.data(), mflags.size());

    // images -> CUDA texture objects (uchar4, point sampling, raw element reads)
    std::vector<uint2> sizes(std::max<uint32_t>(sc->n_images, 1), make_uint2(1, 1));
    std::vector<cudaTextureObject_t> objs(std::max<uint32_t>(sc->n_images, 1), 0);
    for (uint32_t i = 0; i < sc->n_images; ++i) {
        const nrrt_image& im = sc->images[i];
        if (!im.rgb || !im.width || !im.height) {
            ctx->err = "empty image";
            free_scene(ctx);
            return NRRT_ERR_INVALID;
        }
        std::vector<uchar4> rgba((size_t)im.width * im.height);
        for (size_t k = 0; k < rgba.size(); ++k)
            rgba[k] = make_uchar4(im.rgb[3 * k], im.rgb[3 * k + 1], im.rgb[3 * k + 2], 255);
        cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
        cudaArray_t arr = nullptr;
        CK(cudaMallocArray(&arr, &fmt, im.width, im.height));
        ctx->tex_arrays.push_back(arr);
        CK(cudaMemcpy2DToArray(arr, 0, 0, rgba.data(), (size_t)im.width * 4, (size_t)im.width * 4, im.height,
                               cudaMemcpyHostToDevice));
        cudaResourceDesc rd;
        std::memset(&rd, 0, sizeof rd);
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        cudaTextureDesc td;
        std::memset(&td, 0, sizeof td);
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        cudaTextureObject_t to = 0;
        CK(cudaCreateTextureObject(&to, &rd, &td, nullptr));
        ctx->tex_objs.push_back(to);
        objs[i] = to;
        sizes[i] = make_uint2(im.width, im.height);
    }
    UP(image_tex, objs.data(), objs.size());
    UP(image_size, sizes.data(), sizes.size());
#undef UP
    D.n_nodes = sc->n_nodes, D.n_wnodes = sc->n_wnodes, D.n_spheres = sc->n_spheres, D.n_planes = sc->n_planes;
    D.n_instances = sc->n_instances, D.n_materials = sc->n_materials, D.n_textures = sc->n_textures;
    CK(cudaStreamSynchronize(ctx->stream));  // host staging vectors die at return
    {
        uint32_t need = 0;
        if (sc->n_spheres) need |= NRRT_F_SPHERES;
        if (sc->n_planes) need |= NRRT_F_PLANES;
        if (sc->n_instances) need |= NRRT_F_INSTANCES;
        for (uint32_t i = 0; i < sc->n_textures; ++i)
            if (sc->textures[i].kind != NRRT_TEX_SOLID) need |= NRRT_F_TEXTURED;
        for (uint32_t i = 0; i < sc->n_materials; ++i)
            if (sc->materials[i].kind == NRRT_MAT_DIELECTRIC) need |= NRRT_F_DIELECTRIC;
        if (sc->n_spheres && sc->sphere_speed) need |= NRRT_F_MOTION;
        ctx->features = pick_features(need);
        // speculative traversal pays once rays walk more than a handful of nodes (measured: Cornell's 17-node tree
        // loses 4 %, the 487-node sphere field gains 7 %, the 6319-node mesh 16 %)
        ctx->speculate = sc->n_nodes >= NRRT_BINARY_MAX_NODES;
        if (const char* e = std::getenv("NRRT_SPECULATE")) ctx->speculate = std::atoi(e) != 0;  // developer override
        if (!binary_ok) ctx->speculate = true;  // the plain instantiation walks the binary nodes
        ctx->has_binary = binary_ok;
        ctx->binary_stack = binary_ok ? binary_stack_need(sc) + 2 : 0;
    }
    ctx->dev = D;
    ctx->max_stack = sc->max_stack;
    ctx->has_scene = true;
    return NRRT_OK;
}

// Kernel instantiations by scene features (see NRRT_F_* in rt_device.cuh): the three shapes the shipped scenes
// have, plus the general one.
#define NRRT_F_CORNELL (NRRT_F_PLANES | NRRT_F_INSTANCES)                 // planar scenes with wrappers, solid colours
#define NRRT_F_BALLS (NRRT_F_SPHERES | NRRT_F_DIELECTRIC)                  // sphere fields, solid colours
#define NRRT_F_BALLS_TEX (NRRT_F_SPHERES | NRRT_F_TEXTURED)                // textured spheres (earth, noise)
#define NRRT_F_GENERAL (NRRT_F_ALL & ~NRRT_F_MOTION)                       // everything a scene file can describe
static uint32_t pick_features(uint32_t need) {
    for (uint32_t cand : {NRRT_F_CORNELL, NRRT_F_BALLS, NRRT_F_BALLS_TEX, NRRT_F_GENERAL})
        if ((need & ~cand) == 0) return cand;
    return NRRT_F_ALL;
}
static void launch_extend(nrrt_ctx* ctx, unsigned blocks, size_t smem, const WfState& Wf, uint32_t n, uint32_t qin) {
    switch (ctx->features) {
        case NRRT_F_CORNELL: k_wf_extend<NRRT_F_CORNELL><<<blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, Wf, n, qin); break;
        case NRRT_F_BALLS: k_wf_extend<NRRT_F_BALLS><<<blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, Wf, n, qin); break;
        case NRRT_F_BALLS_TEX: k_wf_extend<NRRT_F_BALLS_TEX><<<blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, Wf, n, qin); break;
        case NRRT_F_GENERAL: k_wf_extend<NRRT_F_GENERAL><<<blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, Wf, n, qin); break;
        default: k_wf_extend<NRRT_F_ALL><<<blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, Wf, n, qin); break;
    }
}
static void launch_shade(nrrt_ctx* ctx, unsigned blocks, const nrrt_camera& c, const RenderParams& P, const WfState& Wf,
                         uint32_t qin) {
    switch (ctx->features) {
#define NRRT_SHADE_CASE(FEAT)                                                                                   \
    if (P.active) k_wf_shade<FEAT | NRRT_F_ACTIVE><<<blocks, NRRT_BLOCK, 0, ctx->stream>>>(ctx->dev, c, P, Wf, qin); \
    else k_wf_shade<FEAT><<<blocks, NRRT_BLOCK, 0, ctx->stream>>>(ctx->dev, c, P, Wf, qin);
        case NRRT_F_CORNELL: NRRT_SHADE_CASE(NRRT_F_CORNELL) break;
        case NRRT_F_BALLS: NRRT_SHADE_CASE(NRRT_F_BALLS) break;
        case NRRT_F_BALLS_TEX: NRRT_SHADE_CASE(NRRT_F_BALLS_TEX) break;
        case NRRT_F_GENERAL: NRRT_SHADE_CASE(NRRT_F_GENERAL) break;
        default: NRRT_SHADE_CASE(NRRT_F_ALL) break;
#undef NRRT_SHADE_CASE
    }
}

static cudaError_t launch_fused(nrrt_ctx* ctx, unsigned blocks, const nrrt_camera& c, const RenderParams& P, double* partials) {
    const size_t smem = (size_t)NRRT_BLOCK * (NRRT_STACK_CAP * sizeof(uint32_t) + NRRT_FUSED_STATE_DOUBLES * sizeof(double) +
                                              NRRT_FUSED_STATE_WORDS * sizeof(uint32_t));
    cudaError_t e = cudaSuccess;
#define NRRT_FUSED_LAUNCH(FEAT, MB, SPEC)                                                                              \
    e = cudaFuncSetAttribute(k_render_fused<FEAT, MB, SPEC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
    if (e == cudaSuccess)                                                                                              \
        k_render_fused<FEAT, MB, SPEC><<<blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, c, P, partials, ctx->d_counters);
#define NRRT_FUSED_SPEC(FEAT, MB)                                                                                      \
    if (ctx->speculate) {                                                                                              \
        NRRT_FUSED_LAUNCH(FEAT, MB, true)                                                                              \
    } else {                                                                                                           \
        NRRT_FUSED_LAUNCH(FEAT, MB, false)                                                                             \
    }
#define NRRT_FUSED_CASE(FEAT, MB)                                                                                      \
    if (P.active) {                                                                                                    \
        NRRT_FUSED_SPEC(FEAT | NRRT_F_ACTIVE, MB)                                                                      \
    } else {                                                                                                           \
        NRRT_FUSED_SPEC(FEAT, MB)                                                                                      \
    }
    switch (ctx->features) {
        case NRRT_F_CORNELL: NRRT_FUSED_CASE(NRRT_F_CORNELL, NRRT_FUSED_BLOCKS_PER_SM) break;
        case NRRT_F_BALLS: NRRT_FUSED_CASE(NRRT_F_BALLS, NRRT_FUSED_BLOCKS_PER_SM) break;
        case NRRT_F_BALLS_TEX: NRRT_FUSED_CASE(NRRT_F_BALLS_TEX, NRRT_FUSED_BLOCKS_PER_SM) break;
        case NRRT_F_GENERAL: NRRT_FUSED_CASE(NRRT_F_GENERAL, NRRT_FUSED_BLOCKS_PER_SM) break;
        default: NRRT_FUSED_CASE(NRRT_F_ALL, NRRT_FUSED_BLOCKS_PER_SM) break;
    }
#undef NRRT_FUSED_CASE
#undef NRRT_FUSED_SPEC
#undef NRRT_FUSED_LAUNCH
    return e;
}

// ---- pooled kernel: launch geometry.  Shared memory bounds the slots in flight: pick the warps per block that
// fits the most warps on an SM (each block also costs 1 KB of reserved shared memory).
#ifndef NRRT_POOL_NS
#define NRRT_POOL_NS 64  // path slots per warp
#endif
extern "C++" {
#define NRRT_POOL_STATIC_SMEM 1024  // the opt-in limit covers static + dynamic shared memory; the kernel has 16 B static
struct PoolPlan {
    unsigned warps_per_block = 0, blocks_per_sm = 0;
    size_t smem = 0, cold_bytes_per_slot = 0;
    uint32_t cap = 0;
    uint64_t slots = 0;  // resident path slots on the whole GPU
    bool lite = false;   // the two-stage variant for small scenes (binary nodes, lane-owned traversal)
};
template <uint32_t F, bool LITE>
static PoolPlan pool_plan_f(const nrrt_ctx* ctx) {
    using PL = Pool<F, NRRT_POOL_NS, LITE>;
    PoolPlan best;
    best.lite = LITE;
    // (LITE walks the binary nodes: their stack need is what nrrt_scene_upload computed for them)
    best.cap = std::min<uint32_t>(NRRT_STACK_CAP, (std::max<uint32_t>(LITE ? ctx->binary_stack : ctx->max_stack, 4u) + 3u) & ~3u);
    best.cold_bytes_per_slot = PL::cold_bytes_per_slot();
    const size_t bpw = PL::bytes_per_warp(best.cap);
    unsigned best_warps = 0;
    unsigned force = 0;
    if (const char* e = std::getenv("NRRT_POOL_WPB")) force = (unsigned)std::atoi(e);  // developer override
    for (unsigned wpb = NRRT_POOL_WARPS; wpb >= 1; --wpb) {
        if (force && wpb != force) continue;
        const size_t smem = wpb * bpw;
        if (smem + NRRT_POOL_STATIC_SMEM > ctx->smem_per_block) continue;
        // (the attribute is a per-function limit shared by every host thread: always the device maximum, never a
        // per-launch value another thread's launch could find lowered — nrrt_render_multi renders from several threads)
        if (cudaFuncSetAttribute(k_render_pool<F, NRRT_POOL_NS, LITE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)ctx->smem_per_block - NRRT_POOL_STATIC_SMEM) != cudaSuccess)
            continue;
        int blocks = 0;  // resident blocks per SM: shared memory AND registers
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, k_render_pool<F, NRRT_POOL_NS, LITE>, (int)wpb * 32, smem) != cudaSuccess)
            continue;
        if ((unsigned)blocks * wpb > best_warps) {
            best_warps = (unsigned)blocks * wpb;
            best.warps_per_block = wpb, best.blocks_per_sm = (unsigned)blocks, best.smem = smem;
        }
    }
    (void)cudaGetLastError();
    best.slots = (uint64_t)ctx->sms * best_warps * NRRT_POOL_NS;
    return best;
}
// (active: the instantiations of an adaptive pass, NRRT_F_ACTIVE)
static PoolPlan pool_plan(const nrrt_ctx* ctx, bool lite, bool active) {
#define NRRT_POOL_PLAN(FEAT)                                                                                     \
    if (active) return lite ? pool_plan_f<FEAT | NRRT_F_ACTIVE, true>(ctx) : pool_plan_f<FEAT | NRRT_F_ACTIVE, false>(ctx); \
    return lite ? pool_plan_f<FEAT, true>(ctx) : pool_plan_f<FEAT, false>(ctx);
    switch (ctx->features) {
        case NRRT_F_CORNELL: NRRT_POOL_PLAN(NRRT_F_CORNELL)
        case NRRT_F_BALLS: NRRT_POOL_PLAN(NRRT_F_BALLS)
        case NRRT_F_BALLS_TEX: NRRT_POOL_PLAN(NRRT_F_BALLS_TEX)
        case NRRT_F_GENERAL: NRRT_POOL_PLAN(NRRT_F_GENERAL)
        default: NRRT_POOL_PLAN(NRRT_F_ALL)
    }
#undef NRRT_POOL_PLAN
}
static unsigned pool_blocks(const PoolPlan& pl, uint32_t n_slots) {
    const unsigned per_block = pl.warps_per_block * NRRT_POOL_NS;
    return (unsigned)((n_slots + per_block - 1) / per_block);
}
static cudaError_t launch_pool(nrrt_ctx* ctx, const PoolPlan& pl, const nrrt_camera& c, const RenderParams& P, double* partials,
                               double* cold) {
    if (pl.warps_per_block == 0) return cudaErrorInvalidConfiguration;
    const unsigned blocks = pool_blocks(pl, P.n_slots);
    const uint32_t cold_slots = blocks * pl.warps_per_block * NRRT_POOL_NS;
    cudaError_t e = cudaSuccess;
#define NRRT_POOL_LAUNCH_L(FEAT, LITE)                                                                                    \
    e = cudaFuncSetAttribute(k_render_pool<FEAT, NRRT_POOL_NS, LITE>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                             (int)ctx->smem_per_block - NRRT_POOL_STATIC_SMEM);                                           \
    if (e == cudaSuccess)                                                                                                 \
        k_render_pool<FEAT, NRRT_POOL_NS, LITE><<<blocks, pl.warps_per_block * 32, pl.smem, ctx->stream>>>(               \
            ctx->dev, c, P, partials, ctx->d_counters, pl.cap, cold, cold_slots);
#define NRRT_POOL_LITE(FEAT)                                                                                              \
    if (pl.lite) {                                                                                                        \
        NRRT_POOL_LAUNCH_L(FEAT, true)                                                                                    \
    } else {                                                                                                              \
        NRRT_POOL_LAUNCH_L(FEAT, false)                                                                                   \
    }
#define NRRT_POOL_LAUNCH(FEAT)                                                                                            \
    if (P.active) {                                                                                                       \
        NRRT_POOL_LITE(FEAT | NRRT_F_ACTIVE)                                                                              \
    } else {                                                                                                              \
        NRRT_POOL_LITE(FEAT)                                                                                              \
    }
    switch (ctx->features) {
        case NRRT_F_CORNELL: NRRT_POOL_LAUNCH(NRRT_F_CORNELL) break;
        case NRRT_F_BALLS: NRRT_POOL_LAUNCH(NRRT_F_BALLS) break;
        case NRRT_F_BALLS_TEX: NRRT_POOL_LAUNCH(NRRT_F_BALLS_TEX) break;
        case NRRT_F_GENERAL: NRRT_POOL_LAUNCH(NRRT_F_GENERAL) break;
        default: NRRT_POOL_LAUNCH(NRRT_F_ALL) break;
    }
#undef NRRT_POOL_LAUNCH_L
#undef NRRT_POOL_LITE
#undef NRRT_POOL_LAUNCH
    return e;
}
}  // extern "C++"

static int ensure_scratch(nrrt_ctx* ctx, size_t bytes) {
    if (ctx->scratch_bytes >= bytes) return NRRT_OK;
    if (ctx->scratch) {
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaFree(ctx->scratch));
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
    }
    CK(cudaMalloc(&ctx->scratch, bytes));
    ctx->scratch_bytes = bytes;
    return NRRT_OK;
}

int nrrt_trace_rays(nrrt_ctx* ctx, const double* rays, uint64_t n, double tmin, double tmax, uint32_t flags,
                    nrrt_hit* out, nrrt_trace_stats* stats) {
    if (!ctx) return NRRT_ERR_INVALID;
    if (!ctx->has_scene) {
        ctx->err = "nrrt_trace_rays before nrrt_scene_upload";
        return NRRT_ERR_NO_SCENE;
    }
    if (n == 0) {
        if (stats) std::memset(stats, 0, sizeof *stats);
        return NRRT_OK;
    }
    if (!rays || !out) return NRRT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const bool dev_buf = (flags & NRRT_TRACE_DEVICE_BUFFERS) != 0;
    const size_t hit_bytes = (flags & NRRT_TRACE_COMPACT) ? sizeof(nrrt_hit_compact) : sizeof(nrrt_hit);
    const double* d_rays = rays;
    nrrt_hit* d_out = out;
    if (!dev_buf) {
        size_t rb = (size_t)n * 6 * sizeof(double), hb = (size_t)n * hit_bytes;
        int rc = ensure_scratch(ctx, rb + hb);
        if (rc != NRRT_OK) return rc;
        d_rays = (const double*)ctx->scratch;
        d_out = (nrrt_hit*)((char*)ctx->scratch + rb);
        CK(cudaMemcpyAsync((void*)d_rays, rays, rb, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaMemsetAsync(ctx->d_counters, 0, 8 * sizeof(unsigned long long), ctx->stream));
    dim3 grid((unsigned)((n + NRRT_BLOCK - 1) / NRRT_BLOCK)), block(NRRT_BLOCK);
    size_t smem = (size_t)NRRT_BLOCK * NRRT_STACK_CAP * sizeof(uint32_t);
    const bool count = stats != nullptr && (flags & NRRT_TRACE_COUNT) != 0 && !(flags & NRRT_TRACE_COMPACT);
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (flags & NRRT_TRACE_COMPACT) {
        if (flags & NRRT_TRACE_VISIT_ALL)
            k_trace_rays<true, false, true><<<grid, block, smem, ctx->stream>>>(ctx->dev, d_rays, n, tmin, tmax, ctx->trace_time, d_out, ctx->d_counters);
        else
            k_trace_rays<false, false, true><<<grid, block, smem, ctx->stream>>>(ctx->dev, d_rays, n, tmin, tmax, ctx->trace_time, d_out, ctx->d_counters);
    } else if (flags & NRRT_TRACE_VISIT_ALL) {
        if (count)
            k_trace_rays<true, true><<<grid, block, smem, ctx->stream>>>(ctx->dev, d_rays, n, tmin, tmax, ctx->trace_time, d_out, ctx->d_counters);
        else
            k_trace_rays<true, false><<<grid, block, smem, ctx->stream>>>(ctx->dev, d_rays, n, tmin, tmax, ctx->trace_time, d_out, ctx->d_counters);
    } else {
        if (count)
            k_trace_rays<false, true><<<grid, block, smem, ctx->stream>>>(ctx->dev, d_rays, n, tmin, tmax, ctx->trace_time, d_out, ctx->d_counters);
        else
            k_trace_rays<false, false><<<grid, block, smem, ctx->stream>>>(ctx->dev, d_rays, n, tmin, tmax, ctx->trace_time, d_out, ctx->d_counters);
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    if (!dev_buf) CK(cudaMemcpyAsync(out, d_out, (size_t)n * hit_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long hc[3] = {0, 0, 0};
    if (stats) CK(cudaMemcpyAsync(hc, ctx->d_counters, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (stats) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        stats->node_visits = hc[0];
        stats->box_exact = hc[1];
        stats->prim_tests = hc[2];
        stats->kernel_ms = ms;
    }
    return NRRT_OK;
}

// The chunks of a pixel (see nrrt_render): n_eq equal chunks of `chunk` samples, then halving chunks over the rest.
// Closed form, so the kernels need no table (decode_item).
static void chunk_schedule(uint32_t spp, uint64_t total_pixels, uint32_t& chunk, uint32_t& n_eq, uint32_t& n_chunks) {
    if (spp < 1) spp = 1;
    uint32_t eq_parts = (uint32_t)std::min<uint64_t>(28, std::max<uint64_t>(8, 60000000ull / std::max<uint64_t>(total_pixels, 1)));
    uint32_t tail_shift = 4, tail_max = 0;  // no halving tail by default (see nrrt_render); NRRT_CHUNKS=28,4,4 turns one on
    if (const char* e = std::getenv("NRRT_CHUNKS")) std::sscanf(e, "%u,%u,%u", &eq_parts, &tail_shift, &tail_max);  // developer override
    uint32_t R = tail_max ? (spp >> std::min<uint32_t>(tail_shift, 31)) : 0;   // samples left to the halving tail
    if (eq_parts == 0) R = spp;
    const uint32_t head = spp - R;
    chunk = eq_parts ? std::max<uint32_t>(1, (head + eq_parts - 1) / eq_parts) : 1;
    n_eq = eq_parts ? head / chunk : 0;            // whole equal chunks; what they leave over joins the tail
    R = spp - n_eq * chunk;
    uint32_t n_tail = R ? 1 : 0;
    while (n_tail && n_tail < std::max<uint32_t>(tail_max, 1) && (R >> n_tail) >= 1) ++n_tail;
    n_chunks = n_eq + n_tail;
    if (n_chunks == 0) n_chunks = 1, n_eq = 0;     // spp >= 1 always gives at least one chunk; belt and braces
}

// Work-item layout of a render, for bindings and tests: writes the first sample of every chunk of a pixel and spp as
// the last entry (n_chunks + 1 values, at most `max`); returns n_chunks.  Depends on spp and the image size only.
uint32_t nrrt_chunk_starts(uint32_t samples_per_pixel, uint64_t total_pixels, uint32_t* starts, uint32_t max) {
    const uint32_t spp = std::max<uint32_t>(samples_per_pixel, 1);
    uint32_t chunk = 0, n_eq = 0, n = 0;
    chunk_schedule(spp, total_pixels, chunk, n_eq, n);
    for (uint32_t c = 0; c <= n && starts && c < max; ++c) {
        uint32_t first;
        if (c == n) first = spp;
        else if (c < n_eq) first = c * chunk;
        else {
            const uint32_t base = n_eq * chunk, R = spp - base, k = c - n_eq;
            first = base + R - (R >> k);
        }
        starts[c] = first;
    }
    return n;
}

static uint32_t owned_rows(uint32_t H, uint32_t rank, uint32_t world, uint32_t R) {
    uint32_t rows = 0;
    for (uint32_t b = rank; (uint64_t)b * R < H; b += world) rows += std::min<uint32_t>(R, H - b * R);
    return rows;
}

// Partition and work-item fields of RenderParams (everything decode_item / owned_pixel / item_block_size read, bar the
// slot counts) of a launch over chunks [c0, c1) (c1 clamped to the pixel's chunks): shared by the renders and
// nrrt_work_items / nrrt_pass_items.  With `active` (an adaptive pass) the launch covers the n_active owned pixels it
// lists instead of every owned pixel.  Returns nullptr or the reason it cannot be done.
static const char* work_item_params(RenderParams& P, uint32_t W, uint32_t H, uint32_t spp, uint32_t rank, uint32_t world,
                                    uint32_t rows_per_block, uint32_t c0 = 0, uint32_t c1 = 0xFFFFFFFFu,
                                    const uint32_t* active = nullptr, uint32_t n_active = 0) {
    const uint64_t total_pixels = (uint64_t)W * H;
    P.rank = rank, P.world = world, P.rows_per_block = rows_per_block;
    P.n_owned_pixels = owned_rows(H, rank, world, rows_per_block) * W;
    P.active = active;
    const uint32_t n_pixels = active ? n_active : P.n_owned_pixels;  // pixels of each chunk of the launch
    if (n_pixels > P.n_owned_pixels) return "internal error: more active pixels than owned ones";
    // Work items of a pixel.  They fix the order in which its samples are summed, so they may depend only on what
    // every rank of every partition agrees on — spp and the size of the WHOLE image — never on slots, rank or world:
    // the image is then bit-identical for every slot count and GPU count.  Items are numbered chunk-major (every
    // pixel's chunk 0, then every pixel's chunk 1, ...) and handed to a WARP in blocks of NRRT_ITEM_BLOCK consecutive
    // ones, i.e. consecutive pixels of one chunk (see the kernels).  Measured (profiles/r02_chunk_schedules.log,
    // r02_item_blocks_and_chunk_schedules.log):
    //  * what matters most is that the lanes of a warp stay on neighbouring pixels — same materials, textures and
    //    subtrees.  With one global counter and an item per lane that only held for tiny items (noise.toml: 5552
    //    Mrays/s with 1-sample items, 4798 with 2-sample ones, 4361 with seven halving chunks); with per-warp blocks it
    //    holds for any item size, and every scene gained 6-16 % (Cornell 6242 -> 6640, noise 4840 -> 5622, earth 11602
    //    -> 12850, teapot 2094 -> 2211 at test sizes; 6482 -> 7006 and 2101 -> 2304 at the benchmark sizes);
    //  * the render ENDS waiting for the last slots to finish their item, which is what eight GPUs sharing one image
    //    lose to.  Ending a pixel on a few HALVING chunks (the last 1/16 of its samples as 40, 20, 10, 9) was built for
    //    that and measured: it makes things worse — one rank's share of the benchmark image (tools/rank_time.py) runs at
    //    6520 Mrays/s with the halving tail and 6743 without, the whole image at 6935 either way — so the schedule is
    //    equal chunks only; what does help is shrinking the item BLOCKS towards the end (item_block_size);
    //  * each item costs 24 B of scratch and sets how long the last warps run alone: up to 28 equal chunks for images
    //    up to 2.1 Mpixel, 8 at 4K (1080p x 1024 spp: 27 x 37 + 25; 4K x 4096 spp: 8 items per pixel, 1.6 GB where
    //    round 1 needed 6.4 GB).
    chunk_schedule(spp, total_pixels, P.chunk, P.n_eq, P.n_chunks);
    c1 = std::min(c1, P.n_chunks);
    if (c0 > c1) return "chunk range past the last chunk";
    const uint64_t n_items64 = (uint64_t)n_pixels * (c1 - c0);
    if (n_items64 > 0xFFFFFFF0ull) return "too many work items";
    P.c0 = c0;
    P.n_items = (uint32_t)n_items64;
    P.long_end = (std::min(std::max(P.n_eq, c0), c1) - c0) * n_pixels;  // (fits: n_items does)
    P.n_slots = P.n_warps = 0;
    P.div_pixels = FastDiv::make(n_pixels);
    P.div_rows = FastDiv::make(rows_per_block);
    {
        const uint32_t rows = P.n_owned_pixels / W;
        uint32_t tile_rows = 1;  // largest divisor of rows_per_block that is <= NRRT_TILE_ROWS
        for (uint32_t t = 1; t <= NRRT_TILE_ROWS; ++t)
            if (rows_per_block % t == 0) tile_rows = t;
        if ((uint64_t)W * tile_rows > 0x7FFFFFFFull) return "image too wide";
        P.div_tile = FastDiv::make(tile_rows);
        P.div_strip = FastDiv::make(W * tile_rows);
        P.full_strips = rows / tile_rows;
        P.div_last = FastDiv::make(std::max<uint32_t>(rows % tile_rows, 1));
    }
    for (uint32_t probe : {0u, 1u, W - 1, W, W + 1, P.n_owned_pixels - 1, P.n_owned_pixels, n_pixels - 1, n_pixels,
                           P.n_items - 1, 0x7fffffffu, 0xfffffff0u}) {  // the multiply-shift must agree with '/' (cheap self-check)
        if (P.div_pixels.div(probe) != probe / P.div_pixels.d || P.div_strip.div(probe) != probe / P.div_strip.d ||
            P.div_rows.div(probe) != probe / P.div_rows.d || P.div_last.div(probe) != probe / P.div_last.d ||
            P.div_tile.div(probe) != probe / P.div_tile.d)
            return "internal error: FastDiv self-check failed";
    }
    return nullptr;
}

// Work items [first, first + n) of one rank's launch over chunks [c0, c1) (and the active pixels, see
// work_item_params), decoded by the very functions the kernels use: 4 values per item (x, y, first sample, one past the
// last sample).  Returns the number of items of that launch, 0 if the arguments are not ones the renders would take.
static uint32_t decode_pass(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank, uint32_t world,
                            uint32_t rows_per_block, uint32_t c0, uint32_t c1, const uint32_t* active, uint32_t n_active,
                            uint32_t first, uint32_t n, uint32_t* out) {
    if (width == 0 || height == 0 || (uint64_t)width * height > 0x7FFFFFFFull) return 0;
    if (world == 0) world = 1;
    if (rank >= world) return 0;
    if (rows_per_block == 0) rows_per_block = 8;
    RenderParams P;
    P.key = make_uint2(0, 0);
    nrrt_camera cam;
    std::memset(&cam, 0, sizeof cam);
    cam.width = width, cam.height = height, cam.samples_per_pixel = std::max<uint32_t>(samples_per_pixel, 1);
    if (work_item_params(P, width, height, cam.samples_per_pixel, rank, world, rows_per_block, c0, c1, active, n_active))
        return 0;
    for (uint32_t i = 0; out && i < n && (uint64_t)first + i < P.n_items; ++i) {
        WorkItem wi;
        const uint32_t s0 = active ? decode_item<true>(cam, P, first + i, wi) : decode_item<false>(cam, P, first + i, wi);
        out[4 * i + 0] = wi.x, out[4 * i + 1] = wi.y, out[4 * i + 2] = s0, out[4 * i + 3] = wi.sample_end;
    }
    return P.n_items;
}

uint32_t nrrt_pass_items(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank, uint32_t world,
                         uint32_t rows_per_block, uint32_t c0, uint32_t c1, uint32_t first, uint32_t n, uint32_t* out) {
    return decode_pass(width, height, samples_per_pixel, rank, world, rows_per_block, c0, c1, nullptr, 0, first, n, out);
}

uint32_t nrrt_work_items(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank, uint32_t world,
                         uint32_t rows_per_block, uint32_t first, uint32_t n, uint32_t* out) {
    return nrrt_pass_items(width, height, samples_per_pixel, rank, world, rows_per_block, 0, 0xFFFFFFFFu, first, n, out);
}

// The active list of an adaptive pass: strictly ascending owned-pixel indices, each below n_owned
static bool active_list_ok(const uint32_t* active, uint32_t n_active, uint32_t n_owned) {
    if (n_active && !active) return false;
    for (uint32_t i = 0; i < n_active; ++i)
        if (active[i] >= n_owned || (i && active[i] <= active[i - 1])) return false;
    return true;
}

uint32_t nrrt_pass_items_active(uint32_t width, uint32_t height, uint32_t samples_per_pixel, uint32_t rank,
                                uint32_t world, uint32_t rows_per_block, uint32_t c0, uint32_t c1,
                                const uint32_t* active, uint32_t n_active, uint32_t first, uint32_t n, uint32_t* out) {
    const uint32_t wd = world ? world : 1;
    if (width == 0 || height == 0 || (uint64_t)width * height > 0x7FFFFFFFull || rank >= wd) return 0;
    if (!active_list_ok(active, n_active, owned_rows(height, rank, wd, rows_per_block ? rows_per_block : 8) * width))
        return 0;
    static const uint32_t none = 0;  // a non-null list for n_active = 0: a pass over no pixel, not over all of them
    return decode_pass(width, height, samples_per_pixel, rank, world, rows_per_block, c0, c1, active ? active : &none,
                       n_active, first, n, out);
}

// An adaptive pass of render_chunks: the pixels it renders, and what k_resolve_adaptive and the compaction need
struct AdaptivePass {
    const uint32_t* active;  // n_active ascending owned-pixel indices (device)
    uint32_t n_active;
    AdaptiveState state;
    const uint32_t* starts;  // nrrt_chunk_starts of the frame (device)
    nrrt_adaptive_opts test;
    uint8_t* keep;           // [n_active]
    uint32_t* block_counts;  // [blocks of NRRT_COMPACT_BLOCK over n_active]
    uint32_t* next_active;   // receives the pixels still active after the pass, in order ...
    uint32_t* n_next;        // ... and their count
};

// Renders chunks [c0, c1) of every pixel rank o.rank owns (o.world >= 1, o.rows_per_block >= 1) into the scratch
// partials and resolves them (k_resolve) onto acc (may be null) and, divided by `samples`, into the image *fb (may be
// null; with fb_scratch a full-size image is carved in the scratch and returned in *fb): the body of nrrt_render (all
// chunks) and of nrrt_accum_render (a pass).  An adaptive pass (ad) renders the active pixels only and resolves them
// with k_resolve_adaptive instead, then compacts the active list.  Picks the design, carves the scratch, launches, and
// fills stats.
static int render_chunks(nrrt_ctx* ctx, const nrrt_camera& c, nrrt_render_opts o, uint32_t c0, uint32_t c1, double* acc,
                         double samples, float** fb, bool fb_scratch, bool packed, nrrt_progress_fn progress, void* user,
                         nrrt_render_stats* stats, const char* who, const AdaptivePass* ad = nullptr) {
    const uint32_t W = c.width, H = c.height;
    RenderParams P;
    P.key = make_uint2((uint32_t)o.seed, (uint32_t)(o.seed >> 32));
    if (const char* why = work_item_params(P, W, H, c.samples_per_pixel, o.rank, o.world, o.rows_per_block, c0, c1,
                                           ad ? ad->active : nullptr, ad ? ad->n_active : 0)) {
        ctx->err = std::string(who) + ": " + why;
        return std::strstr(why, "internal") ? NRRT_ERR_INVALID : NRRT_ERR_LIMIT;
    }
    const uint64_t n_items64 = P.n_items;
    const uint32_t want_slots = o.max_slots ? o.max_slots : (1u << 21);
    P.n_slots = (uint32_t)std::min<uint64_t>(n_items64, want_slots);

    const bool counting = (o.flags & NRRT_RENDER_COUNT) != 0;
    // NRRT_MODE_AUTO: the pooled kernel wins where rays walk many nodes (measured on B200: 6319-node teapot 2045 vs
    // 1391 Mrays/s, Cornell box + teapot 1894 vs 1480) and loses where shading dominates (487-node sphere field 4209 vs
    // 4557, Cornell box 3735 vs 6161), so the split is by tree size
    if (o.mode == NRRT_MODE_AUTO) {
        o.mode = ctx->dev.n_nodes >= NRRT_POOL_MIN_NODES ? NRRT_MODE_POOL : NRRT_MODE_FUSED;
        if (const char* e = std::getenv("NRRT_AUTO_MODE")) o.mode = (uint32_t)std::atoi(e);  // developer override
    }
    if (o.mode > NRRT_MODE_POOL) {
        ctx->err = std::string(who) + ": unknown mode";
        return NRRT_ERR_INVALID;
    }
    // (instance chains are packed as 16-bit indices in the pooled kernel's slot state: larger scenes use the fused kernel)
    const bool pooled = o.mode == NRRT_MODE_POOL && !counting && ctx->dev.n_instances <= 65536u;
    if (o.mode == NRRT_MODE_POOL && !counting && !pooled) o.mode = NRRT_MODE_FUSED;
    const bool wavefront = o.mode == NRRT_MODE_WAVEFRONT && !counting;
    const bool fused = o.mode == NRRT_MODE_FUSED && !counting;

    PoolPlan plan;
    if (pooled) {  // persistent: every resident pool slot starts with one item; the work counter hands out the rest
        // small scenes (binary nodes on the device): the two-stage variant
        bool lite = ctx->has_binary;
        if (const char* e = std::getenv("NRRT_POOL_LITE")) lite = std::atoi(e) != 0 && ctx->has_binary;  // developer override
        plan = pool_plan(ctx, lite, P.active != nullptr);
        if (plan.warps_per_block == 0) {
            ctx->err = "pooled kernel: the slot pool does not fit in shared memory";
            return NRRT_ERR_LIMIT;
        }
        P.n_slots = (uint32_t)std::min<uint64_t>(n_items64, o.max_slots ? std::min<uint64_t>(o.max_slots, plan.slots) : plan.slots);
    }
    if (fused) {  // persistent: one thread per resident lane; the work counter hands out the rest
        const uint64_t resident = (uint64_t)(ctx->persistent_blocks / NRRT_EXTEND_MINBLOCKS) * NRRT_FUSED_BLOCKS_PER_SM * NRRT_BLOCK;
        P.n_slots = (uint32_t)std::min<uint64_t>(n_items64, o.max_slots ? std::min<uint64_t>(o.max_slots, resident) : resident);
    }
    P.n_warps = pooled ? (P.n_slots + NRRT_POOL_NS - 1) / NRRT_POOL_NS : (P.n_slots + 31) / 32;
    const size_t fb_bytes = (size_t)W * H * 3 * sizeof(float);
    const size_t n = P.n_slots;
    // scratch layout
    size_t off = 0;
    auto carve = [&](size_t bytes) {
        size_t at = off;
        off += (bytes + 255) & ~(size_t)255;
        return at;
    };
    size_t o_fb = fb_scratch ? carve(fb_bytes) : 0;
    size_t o_part = carve((size_t)P.n_items * 3 * sizeof(double));
    size_t o_cold = 0;
    if (pooled) {
        const size_t cold_slots = (size_t)pool_blocks(plan, P.n_slots) * plan.warps_per_block * NRRT_POOL_NS;
        o_cold = carve(cold_slots * plan.cold_bytes_per_slot);
    }
    size_t o_ray = 0, o_T = 0, o_sum = 0, o_attr = 0, o_item = 0, o_sample = 0, o_bounce = 0, o_ht = 0, o_hp = 0, o_hi = 0,
           o_q0 = 0, o_q1 = 0, o_cnt = 0;
    if (wavefront) {
        o_ray = carve(n * 7 * sizeof(double));
        o_T = carve(n * 3 * sizeof(double));
        o_sum = carve(n * 3 * sizeof(double));
        o_item = carve(n * sizeof(uint32_t));
        o_sample = carve(n * sizeof(uint32_t));
        o_bounce = carve(n * sizeof(uint32_t));
        o_ht = carve(n * sizeof(double));
        o_hp = carve(n * sizeof(uint32_t));
        o_hi = carve(n * NRRT_MAX_INSTANCE_DEPTH * sizeof(uint32_t));
        o_attr = carve(n * 8 * sizeof(double));
        o_q0 = carve(n * sizeof(uint32_t));
        o_q1 = carve(n * sizeof(uint32_t));
        o_cnt = carve(8 * sizeof(uint32_t));
    }
    if (off > ctx->scratch_bytes) {  // say what is needed instead of failing inside cudaMalloc
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && off > free_b + ctx->scratch_bytes) {
            ctx->err = std::string(who) + ": needs " + std::to_string(off >> 20) + " MiB of device scratch (" +
                       std::to_string(P.n_items) + " work items x 24 B" + (fb_scratch ? " + framebuffer" : "") + "), " +
                       std::to_string((free_b + ctx->scratch_bytes) >> 20) + " MiB available";
            return NRRT_ERR_LIMIT;
        }
    }
    int rc = ensure_scratch(ctx, std::max<size_t>(off, 256));
    if (rc != NRRT_OK) return rc;
    char* base = (char*)ctx->scratch;
    if (fb_scratch) *fb = (float*)(base + o_fb);
    float* d_fb = fb ? *fb : nullptr;
    double* d_part = (double*)(base + o_part);

    // counters: [0] segments [1] paths [2..4] instrumentation [5] next work item (first n_slots pre-assigned)
    unsigned long long init_counters[8] = {0, 0, 0, 0, 0, P.n_slots, 0, 0};
    CK(cudaMemcpyAsync(ctx->d_counters, init_counters, sizeof init_counters, cudaMemcpyHostToDevice, ctx->stream));
    uint64_t launches = 0, extend_launches = 0;
    double extend_ms = 0.0;
    const size_t smem = (size_t)NRRT_BLOCK * NRRT_STACK_CAP * sizeof(uint32_t);
    const unsigned work_blocks = (unsigned)((n + NRRT_BLOCK - 1) / NRRT_BLOCK);
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (n == 0 || c.ray_max_bounces == 0) {
        // nothing owned, or every path returns black at depth 0 (camera.rs:276-278)
        if (P.n_items) CK(cudaMemsetAsync(d_part, 0, (size_t)P.n_items * 3 * sizeof(double), ctx->stream));
    } else if (pooled) {
        CK(launch_pool(ctx, plan, c, P, d_part, (double*)(base + o_cold)));
        CK(cudaGetLastError());
        ++launches;
    } else if (fused) {
        CK(launch_fused(ctx, work_blocks, c, P, d_part));
        CK(cudaGetLastError());
        ++launches;
    } else if (!wavefront) {
        if (counting && P.active)
            k_render_mega<true, true><<<work_blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, c, P, d_part, ctx->d_counters);
        else if (counting)
            k_render_mega<true, false><<<work_blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, c, P, d_part, ctx->d_counters);
        else if (P.active)
            k_render_mega<false, true><<<work_blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, c, P, d_part, ctx->d_counters);
        else
            k_render_mega<false, false><<<work_blocks, NRRT_BLOCK, smem, ctx->stream>>>(ctx->dev, c, P, d_part, ctx->d_counters);
        CK(cudaGetLastError());
        ++launches;
    } else {
        WfState Wf;
        Wf.ray = (double*)(base + o_ray);
        Wf.T = (double*)(base + o_T);
        Wf.sum = (double*)(base + o_sum);
        Wf.item = (uint32_t*)(base + o_item);
        Wf.sample = (uint32_t*)(base + o_sample);
        Wf.bounce = (uint32_t*)(base + o_bounce);
        Wf.hit_t = (double*)(base + o_ht);
        Wf.hit_prim = (uint32_t*)(base + o_hp);
        Wf.hit_inst = (uint32_t*)(base + o_hi);
        Wf.hit_attr = (double*)(base + o_attr);
        Wf.queue[0] = (uint32_t*)(base + o_q0);
        Wf.queue[1] = (uint32_t*)(base + o_q1);
        Wf.count = (uint32_t*)(base + o_cnt);
        Wf.cursor = Wf.count + 4;
        Wf.partials = d_part;
        Wf.counters = ctx->d_counters;
        if (P.active) k_wf_init<true><<<work_blocks, NRRT_BLOCK, 0, ctx->stream>>>(c, P, Wf);
        else k_wf_init<false><<<work_blocks, NRRT_BLOCK, 0, ctx->stream>>>(c, P, Wf);
        CK(cudaGetLastError());
        ++launches;
        // the queue length lives on the device; the host polls it through a pinned ring without stalling
        const int RING = 32, POLL_EVERY = 8, MAX_TIMED = 256;
        while (ctx->ev_pool.size() < (size_t)RING + 2 * MAX_TIMED) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            ctx->ev_pool.push_back(e);
        }
        for (int k = 0; k < 2 * RING; ++k) ctx->h_count[k] = 0x7FFFFFFFu;
        uint64_t iter = 0, polls_issued = 0, polls_seen = 0;
        // expected iteration count, to spread the timed extend launches over the whole render
        const uint64_t expect_iters = std::max<uint64_t>(1, (uint64_t)P.n_items * P.chunk * 4 / std::max<uint32_t>(P.n_slots, 1u));
        const uint64_t time_every = std::max<uint64_t>(1, expect_iters / MAX_TIMED);
        std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timing;
        bool done = false;
        uint32_t qin = 0;
        const uint64_t hard_cap = ((uint64_t)P.n_items * P.chunk / std::max<uint32_t>(P.n_slots, 1u) + P.chunk + 2) *
                                      (uint64_t)c.ray_max_bounces + 64;
        while (!done && iter < hard_cap) {
            bool timed = (iter % time_every == 0) && (int)timing.size() < MAX_TIMED;
            cudaEvent_t ta = nullptr, tb = nullptr;
            if (timed) {
                ta = ctx->ev_pool[RING + 2 * timing.size()], tb = ctx->ev_pool[RING + 2 * timing.size() + 1];
                CK(cudaEventRecord(ta, ctx->stream));
            }
            launch_extend(ctx, std::min<unsigned>(work_blocks, ctx->persistent_blocks), smem, Wf, (uint32_t)n, qin);
            if (timed) {
                CK(cudaEventRecord(tb, ctx->stream));
                timing.emplace_back(ta, tb);
            }
            launch_shade(ctx, work_blocks, c, P, Wf, qin);
            CK(cudaGetLastError());
            launches += 2;
            ++extend_launches;
            qin ^= 1;
            ++iter;
            if (iter % POLL_EVERY == 0) {
                // throttle: never run more than RING polls ahead of the device
                while (polls_issued - polls_seen >= (uint64_t)RING) {
                    CK(cudaEventSynchronize(ctx->ev_pool[polls_seen % RING]));
                    if (ctx->h_count[2 * (polls_seen % RING)] + ctx->h_count[2 * (polls_seen % RING) + 1] == 0) done = true;
                    ++polls_seen;
                }
                int slot = (int)(polls_issued % RING);
                CK(cudaMemcpyAsync(&ctx->h_count[2 * slot], Wf.count + 2 * qin, 2 * sizeof(uint32_t),
                                   cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaEventRecord(ctx->ev_pool[slot], ctx->stream));
                ++polls_issued;
                while (polls_seen < polls_issued && cudaEventQuery(ctx->ev_pool[polls_seen % RING]) == cudaSuccess) {
                    if (ctx->h_count[2 * (polls_seen % RING)] + ctx->h_count[2 * (polls_seen % RING) + 1] == 0) done = true;
                    ++polls_seen;
                }
                // once the queue is nearly drained, wait for each poll instead of launching empty passes
                if (!done && polls_seen > 0 &&
                    ctx->h_count[2 * ((polls_seen - 1) % RING)] + ctx->h_count[2 * ((polls_seen - 1) % RING) + 1] < 4096u) {
                    while (polls_seen < polls_issued) {
                        CK(cudaEventSynchronize(ctx->ev_pool[polls_seen % RING]));
                        if (ctx->h_count[2 * (polls_seen % RING)] + ctx->h_count[2 * (polls_seen % RING) + 1] == 0) done = true;
                        ++polls_seen;
                    }
                }
            }
        }
        CK(cudaStreamSynchronize(ctx->stream));
        double sampled = 0.0;
        for (auto& pr : timing) {
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, pr.first, pr.second));
            sampled += ms;
        }
        if (!timing.empty()) extend_ms = sampled / (double)timing.size() * (double)extend_launches;
    }
    if (ad) {
        if (ad->n_active) {
            const uint32_t blocks = (ad->n_active + NRRT_COMPACT_BLOCK - 1) / NRRT_COMPACT_BLOCK;
            k_resolve_adaptive<<<blocks, NRRT_COMPACT_BLOCK, 0, ctx->stream>>>(c, P, ad->n_active, d_part, ad->state,
                                                                               ad->starts, P.c0 + P.n_items / ad->n_active,
                                                                               ad->test, ad->keep);
            k_compact_count<<<blocks, NRRT_COMPACT_BLOCK, 0, ctx->stream>>>(ad->keep, ad->n_active, ad->block_counts);
            k_compact_scan<<<1, 1024, 0, ctx->stream>>>(ad->block_counts, blocks, ad->n_next);
            k_compact_scatter<<<blocks, NRRT_COMPACT_BLOCK, 0, ctx->stream>>>(ad->active, ad->keep, ad->n_active,
                                                                              ad->block_counts, ad->next_active);
            CK(cudaGetLastError());
            launches += 4;
        }
    } else if (P.n_owned_pixels) {
        k_resolve<<<(P.n_owned_pixels + 255) / 256, 256, 0, ctx->stream>>>(c, P, d_part, acc, samples, d_fb, packed);
        CK(cudaGetLastError());
        ++launches;
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    if (progress && !wavefront && n != 0 && c.ray_max_bounces != 0) {
        // (before the image copy below: a copy into pageable host memory blocks until the render is done)
        // The single-launch kernels hand work items out from a device counter: read it from a side stream while the
        // render runs and report the pixels whose items have all been handed out (render.rs:48-59 ticks once per pixel).
        if (!ctx->side) CK(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
        unsigned long long* h_next = reinterpret_cast<unsigned long long*>(ctx->h_count);  // pinned
        uint64_t last = 0;
        while (cudaEventQuery(ctx->ev1) == cudaErrorNotReady) {
            CK(cudaMemcpyAsync(h_next, ctx->d_counters + 5, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->side));
            CK(cudaStreamSynchronize(ctx->side));
            const uint64_t handed = *h_next > P.n_slots ? *h_next - P.n_slots : 0;  // the last n_slots are still in flight
            const uint64_t done = std::min<uint64_t>(handed, P.n_items) * P.n_owned_pixels / std::max<uint32_t>(P.n_items, 1u);
            if (done > last && done < P.n_owned_pixels) {
                progress(done, P.n_owned_pixels, user);
                last = done;
            }
            std::this_thread::sleep_for(std::chrono::milliseconds(20));
        }
    }
    unsigned long long hc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    CK(cudaMemcpyAsync(hc, ctx->d_counters, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (stats) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        stats->paths = hc[1];
        stats->segments = hc[0];
        stats->launches = launches;
        stats->device_ms = ms;
        stats->extend_ms = wavefront ? extend_ms : ms;
        stats->extend_launches = wavefront ? extend_launches : (launches ? 1 : 0);
        stats->pixels = ad ? ad->n_active : P.n_owned_pixels;
        stats->mode = counting ? (uint32_t)NRRT_MODE_MEGAKERNEL : o.mode;
        stats->node_visits = hc[2];
        stats->box_exact = hc[3];
        stats->prim_tests = hc[4];
        stats->inst_entries = hc[6];
        stats->inst_misses = hc[7];
    }
    return NRRT_OK;
}

// The rows rank o.rank owns, from the device image d_fb (full-size, or packed; px_bytes per pixel) to the caller's host
// buffer.
static int copy_owned_rows(nrrt_ctx* ctx, const nrrt_render_opts& o, uint32_t W, uint32_t H, bool packed,
                           const void* d_fb, void* out_rgb, size_t px_bytes = 3 * sizeof(float)) {
    const uint32_t R = o.rows_per_block;
    const size_t row_bytes = (size_t)W * px_bytes;
    if (packed) {
        const size_t rows = owned_rows(H, o.rank, o.world, R);
        if (rows) CK(cudaMemcpyAsync(out_rgb, d_fb, rows * row_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    } else if (o.world == 1) {  // one contiguous copy
        CK(cudaMemcpyAsync(out_rgb, d_fb, (size_t)H * row_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
        // the owned row-blocks sit at a fixed pitch: one strided copy for the full blocks, one for a cut-off last one
        size_t full_blocks = 0, tail_y0 = 0, tail_rows = 0;
        for (uint32_t b = o.rank; (uint64_t)b * R < H; b += o.world) {
            const size_t y0 = (size_t)b * R, rows = std::min<size_t>(R, H - y0);
            if (rows == R) ++full_blocks;
            else tail_y0 = y0, tail_rows = rows;
        }
        const size_t off0 = (size_t)o.rank * R * row_bytes, pitch = (size_t)o.world * R * row_bytes;
        if (full_blocks)
            CK(cudaMemcpy2DAsync((char*)out_rgb + off0, pitch, (const char*)d_fb + off0, pitch, R * row_bytes, full_blocks,
                                 cudaMemcpyDeviceToHost, ctx->stream));
        if (tail_rows)
            CK(cudaMemcpyAsync((char*)out_rgb + tail_y0 * row_bytes, (const char*)d_fb + tail_y0 * row_bytes,
                               tail_rows * row_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return NRRT_OK;
}

// nrrt_render_opts with the defaults filled in, or the reason they cannot be used
static const char* default_opts(const nrrt_render_opts* in, nrrt_render_opts& o) {
    std::memset(&o, 0, sizeof o);
    if (in) o = *in;
    if (o.world == 0) o.world = 1;
    if (o.rank >= o.world) return "rank >= world";
    if (o.rows_per_block == 0) o.rows_per_block = 8;
    return nullptr;
}

int nrrt_render(nrrt_ctx* ctx, const nrrt_camera* cam, const nrrt_render_opts* opts_in, float* out_rgb,
                nrrt_progress_fn progress, void* user, nrrt_render_stats* stats) {
    if (!ctx) return NRRT_ERR_INVALID;
    if (!ctx->has_scene) {
        ctx->err = "nrrt_render before nrrt_scene_upload";
        return NRRT_ERR_NO_SCENE;
    }
    if (!cam || !out_rgb || cam->width == 0 || cam->height == 0) {
        ctx->err = "nrrt_render: bad camera or output pointer";
        return NRRT_ERR_INVALID;
    }
    nrrt_render_opts o;
    if (const char* why = default_opts(opts_in, o)) {
        ctx->err = std::string("nrrt_render: ") + why;
        return NRRT_ERR_INVALID;
    }
    CK(cudaSetDevice(ctx->device));
    if ((uint64_t)cam->width * cam->height > 0x7FFFFFFFull) {
        ctx->err = "image too large";
        return NRRT_ERR_LIMIT;
    }
    nrrt_camera c = *cam;
    if (c.samples_per_pixel < 1) c.samples_per_pixel = 1;  // camera.rs:104
    const bool out_dev = (o.flags & NRRT_RENDER_OUT_DEVICE) != 0;
    const bool packed = (o.flags & NRRT_RENDER_OUT_PACKED) != 0;
    float* d_fb = out_dev ? out_rgb : nullptr;
    nrrt_render_stats st;
    int rc = render_chunks(ctx, c, o, 0, 0xFFFFFFFFu, nullptr, (double)c.samples_per_pixel, &d_fb, !out_dev, packed,
                           progress, user, &st, "nrrt_render");
    if (rc != NRRT_OK) return rc;
    if (!out_dev && (rc = copy_owned_rows(ctx, o, c.width, c.height, packed, d_fb, out_rgb)) != NRRT_OK) return rc;
    if (progress) progress(st.pixels, st.pixels, user);
    if (stats) *stats = st;
    return NRRT_OK;
}

// ---- progressive rendering: one frame rendered in passes of whole chunks, summed into a persistent f64 accumulator
struct nrrt_accum {
    nrrt_ctx* ctx = nullptr;
    nrrt_camera cam;                // samples_per_pixel >= 1
    nrrt_render_opts opts;          // defaults filled in; flags: NRRT_RENDER_COUNT at most
    uint64_t scene_gen = 0;         // the context's scene this frame belongs to
    std::vector<uint32_t> starts;   // nrrt_chunk_starts: n_chunks + 1 values
    uint32_t chunks_done = 0;
    size_t n_sums = 0;              // 3 x owned pixels
    double* d_sum = nullptr;        // running per-pixel sums, owned rows packed: [j][x][3]
    // adaptive frames only (nrrt_accum_create_adaptive)
    bool adaptive = false;
    nrrt_adaptive_opts test;
    uint32_t n_active = 0;          // pixels still active (every owned pixel before the first pass)
    uint32_t cur = 0;               // d_active[cur] is the active list; a pass compacts it into the other one
    void* d_ad = nullptr;           // one allocation for everything below
    AdaptiveState st;               // S = d_sum; Q, N, K
    uint32_t* d_active[2] = {nullptr, nullptr};
    uint8_t* d_keep = nullptr;      // [owned pixels]: k_resolve_adaptive's verdicts
    uint32_t* d_blocks = nullptr;   // compaction block counts
    uint32_t* d_n_next = nullptr;   // compaction result count
    uint32_t* d_starts = nullptr;   // starts on the device
};

// the accumulator's context is usable and still holds the scene the accumulator was created for
static int accum_check(const nrrt_accum* a, const char* who) {
    if (!a || !a->ctx) return NRRT_ERR_INVALID;
    nrrt_ctx* ctx = a->ctx;
    if (!ctx->has_scene || ctx->scene_gen != a->scene_gen) {
        ctx->err = std::string(who) + ": the context's scene was replaced after nrrt_accum_create";
        return NRRT_ERR_NO_SCENE;
    }
    CK(cudaSetDevice(ctx->device));
    return NRRT_OK;
}

static void accum_release(nrrt_accum* a) {
    if (a->d_sum) cudaFree(a->d_sum);
    if (a->d_ad) cudaFree(a->d_ad);
    delete a;
}

// the body of nrrt_accum_create and nrrt_accum_create_adaptive (test: null for a plain progressive frame)
static int accum_create(nrrt_ctx* ctx, const nrrt_camera* cam, const nrrt_render_opts* opts_in,
                        const nrrt_adaptive_opts* test, nrrt_accum** out, const char* who) {
    if (!ctx || !out) return NRRT_ERR_INVALID;
    *out = nullptr;
    if (!ctx->has_scene) {
        ctx->err = std::string(who) + " before nrrt_scene_upload";
        return NRRT_ERR_NO_SCENE;
    }
    if (!cam || cam->width == 0 || cam->height == 0) {
        ctx->err = std::string(who) + ": bad camera";
        return NRRT_ERR_INVALID;
    }
    nrrt_render_opts o;
    if (const char* why = default_opts(opts_in, o)) {
        ctx->err = std::string(who) + ": " + why;
        return NRRT_ERR_INVALID;
    }
    if (o.mode > NRRT_MODE_AUTO) {
        ctx->err = std::string(who) + ": unknown mode";
        return NRRT_ERR_INVALID;
    }
    if (test && !(std::isfinite(test->rel_error) && test->rel_error >= 0.0 && std::isfinite(test->abs_error) &&
                  test->abs_error >= 0.0)) {
        ctx->err = std::string(who) + ": rel_error and abs_error must be finite and >= 0";
        return NRRT_ERR_INVALID;
    }
    o.flags &= NRRT_RENDER_COUNT;  // the output flags belong to nrrt_accum_image
    if ((uint64_t)cam->width * cam->height > 0x7FFFFFFFull) {
        ctx->err = "image too large";
        return NRRT_ERR_LIMIT;
    }
    CK(cudaSetDevice(ctx->device));
    nrrt_accum* a = new nrrt_accum;
    a->ctx = ctx;
    a->cam = *cam;
    if (a->cam.samples_per_pixel < 1) a->cam.samples_per_pixel = 1;  // camera.rs:104
    a->opts = o;
    a->scene_gen = ctx->scene_gen;
    a->starts.resize(64);
    const uint32_t n_chunks = nrrt_chunk_starts(a->cam.samples_per_pixel, (uint64_t)cam->width * cam->height,
                                                a->starts.data(), (uint32_t)a->starts.size());
    a->starts.resize(n_chunks + 1);
    a->n_sums = (size_t)owned_rows(cam->height, o.rank, o.world, o.rows_per_block) * cam->width * 3;
    const size_t bytes = std::max<size_t>(a->n_sums, 1) * sizeof(double);
    cudaError_t e = cudaMalloc((void**)&a->d_sum, bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->d_sum, 0, bytes, ctx->stream);
    if (e == cudaSuccess && test) {
        a->adaptive = true;
        a->test = *test;
        const size_t n = std::max<size_t>(a->n_sums / 3, 1), blocks = (n + NRRT_COMPACT_BLOCK - 1) / NRRT_COMPACT_BLOCK;
        size_t off = 0;
        auto carve = [&](size_t b) {
            size_t at = off;
            off += (b + 255) & ~(size_t)255;
            return at;
        };
        const size_t o_q = carve(n * 3 * sizeof(double)), o_n = carve(n * 4), o_k = carve(n * 4), o_a0 = carve(n * 4),
                     o_a1 = carve(n * 4), o_keep = carve(n), o_blk = carve(blocks * 4), o_cnt = carve(4),
                     o_st = carve(a->starts.size() * 4);
        e = cudaMalloc(&a->d_ad, off);
        if (e == cudaSuccess) e = cudaMemsetAsync(a->d_ad, 0, off, ctx->stream);
        if (e == cudaSuccess) {
            char* base = (char*)a->d_ad;
            a->st = AdaptiveState{a->d_sum, (double*)(base + o_q), (uint32_t*)(base + o_n), (uint32_t*)(base + o_k)};
            a->d_active[0] = (uint32_t*)(base + o_a0), a->d_active[1] = (uint32_t*)(base + o_a1);
            a->d_keep = (uint8_t*)(base + o_keep);
            a->d_blocks = (uint32_t*)(base + o_blk);
            a->d_n_next = (uint32_t*)(base + o_cnt);
            a->d_starts = (uint32_t*)(base + o_st);
            a->n_active = (uint32_t)(a->n_sums / 3);
            e = cudaMemcpyAsync(a->d_starts, a->starts.data(), a->starts.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
            if (e == cudaSuccess && a->n_active) {
                k_iota<<<(a->n_active + 255) / 256, 256, 0, ctx->stream>>>(a->d_active[0], a->n_active);
                e = cudaGetLastError();
            }
        }
    }
    if (e != cudaSuccess) {
        ctx->err = std::string(who) + ": " + cudaGetErrorString(e);
        accum_release(a);
        return NRRT_ERR_CUDA;
    }
    *out = a;
    return NRRT_OK;
}

int nrrt_accum_create(nrrt_ctx* ctx, const nrrt_camera* cam, const nrrt_render_opts* opts_in, nrrt_accum** out) {
    return accum_create(ctx, cam, opts_in, nullptr, out, "nrrt_accum_create");
}

int nrrt_accum_create_adaptive(nrrt_ctx* ctx, const nrrt_camera* cam, const nrrt_render_opts* opts_in,
                               const nrrt_adaptive_opts* adaptive, nrrt_accum** out) {
    if (!adaptive) {
        if (ctx) ctx->err = "nrrt_accum_create_adaptive: NULL adaptive options";
        if (out) *out = nullptr;
        return NRRT_ERR_INVALID;
    }
    return accum_create(ctx, cam, opts_in, adaptive, out, "nrrt_accum_create_adaptive");
}

int nrrt_accum_render(nrrt_accum* a, uint32_t min_samples, nrrt_render_stats* stats) {
    int rc = accum_check(a, "nrrt_accum_render");
    if (rc != NRRT_OK) return rc;
    const uint32_t n_chunks = (uint32_t)a->starts.size() - 1;
    uint32_t c1 = a->chunks_done;
    while (c1 < n_chunks && a->starts[c1] < min_samples) ++c1;  // whole chunks, up to spp
    nrrt_render_stats st;
    std::memset(&st, 0, sizeof st);
    st.pixels = a->adaptive ? a->n_active : (uint32_t)(a->n_sums / 3);
    if (c1 > a->chunks_done && (!a->adaptive || a->n_active)) {  // (an adaptive frame with no active pixel is done)
        AdaptivePass ap;
        if (a->adaptive)
            ap = AdaptivePass{a->d_active[a->cur], a->n_active, a->st, a->d_starts, a->test, a->d_keep, a->d_blocks,
                              a->d_active[a->cur ^ 1], a->d_n_next};
        rc = render_chunks(a->ctx, a->cam, a->opts, a->chunks_done, c1, a->d_sum, 0.0, nullptr, false, false, nullptr,
                           nullptr, &st, "nrrt_accum_render", a->adaptive ? &ap : nullptr);
        if (rc != NRRT_OK) return rc;
        if (a->adaptive) {  // the only value of the compaction the host needs: 4 bytes per pass
            nrrt_ctx* ctx = a->ctx;
            CK(cudaMemcpyAsync(&a->n_active, a->d_n_next, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            a->cur ^= 1;
        }
        a->chunks_done = c1;
    }
    if (stats) *stats = st;
    return NRRT_OK;
}

uint32_t nrrt_accum_samples(const nrrt_accum* a) { return a ? a->starts[a->chunks_done] : 0; }

uint32_t nrrt_accum_active(const nrrt_accum* a) { return a && a->adaptive ? a->n_active : 0; }

// One of an adaptive frame's per-pixel outputs (k_adaptive_map<what>), laid out as nrrt_accum_image lays out the image
static int adaptive_map(nrrt_accum* a, int what, void* out, uint32_t flags, const char* who) {
    int rc = accum_check(a, who);
    if (rc != NRRT_OK) return rc;
    nrrt_ctx* ctx = a->ctx;
    if (!a->adaptive || !out) {
        ctx->err = std::string(who) + (out ? ": not an adaptive frame (nrrt_accum_create_adaptive)" : ": NULL output");
        return NRRT_ERR_INVALID;
    }
    const nrrt_camera& c = a->cam;
    const nrrt_render_opts& o = a->opts;
    RenderParams P;  // owned_pixel's fields
    P.key = make_uint2(0, 0);
    if (const char* why = work_item_params(P, c.width, c.height, c.samples_per_pixel, o.rank, o.world, o.rows_per_block,
                                           a->chunks_done, a->chunks_done)) {
        ctx->err = std::string(who) + ": " + why;
        return NRRT_ERR_INVALID;
    }
    const size_t px_bytes = what == AMAP_SAMPLES ? sizeof(uint32_t) : 3 * sizeof(float);
    const bool out_dev = (flags & NRRT_RENDER_OUT_DEVICE) != 0, packed = (flags & NRRT_RENDER_OUT_PACKED) != 0;
    void* d_out = out;
    if (!out_dev) {
        if ((rc = ensure_scratch(ctx, std::max<size_t>((size_t)c.width * c.height * px_bytes, 256))) != NRRT_OK) return rc;
        d_out = ctx->scratch;
    }
    if (P.n_owned_pixels) {
        const unsigned blocks = (P.n_owned_pixels + 255) / 256;
        if (what == AMAP_IMAGE) k_adaptive_map<AMAP_IMAGE><<<blocks, 256, 0, ctx->stream>>>(c, P, a->st, d_out, packed);
        else if (what == AMAP_ERROR) k_adaptive_map<AMAP_ERROR><<<blocks, 256, 0, ctx->stream>>>(c, P, a->st, d_out, packed);
        else k_adaptive_map<AMAP_SAMPLES><<<blocks, 256, 0, ctx->stream>>>(c, P, a->st, d_out, packed);
        CK(cudaGetLastError());
    }
    if (out_dev) {
        CK(cudaStreamSynchronize(ctx->stream));
        return NRRT_OK;
    }
    return copy_owned_rows(ctx, o, c.width, c.height, packed, d_out, out, px_bytes);
}

int nrrt_accum_image(nrrt_accum* a, float* out_rgb, uint32_t flags) {
    int rc = accum_check(a, "nrrt_accum_image");
    if (rc != NRRT_OK) return rc;
    nrrt_ctx* ctx = a->ctx;
    if (!out_rgb || a->chunks_done == 0) {
        ctx->err = out_rgb ? "nrrt_accum_image: no samples rendered yet" : "nrrt_accum_image: NULL output";
        return NRRT_ERR_INVALID;
    }
    if (a->adaptive) return adaptive_map(a, AMAP_IMAGE, out_rgb, flags, "nrrt_accum_image");  // each pixel by its own N
    const nrrt_camera& c = a->cam;
    const nrrt_render_opts& o = a->opts;
    RenderParams P;  // owned_pixel's fields; no chunks: k_resolve divides the sums as they are
    P.key = make_uint2(0, 0);
    if (const char* why = work_item_params(P, c.width, c.height, c.samples_per_pixel, o.rank, o.world, o.rows_per_block,
                                           a->chunks_done, a->chunks_done)) {
        ctx->err = std::string("nrrt_accum_image: ") + why;
        return NRRT_ERR_INVALID;
    }
    const bool out_dev = (flags & NRRT_RENDER_OUT_DEVICE) != 0, packed = (flags & NRRT_RENDER_OUT_PACKED) != 0;
    float* d_fb = out_rgb;
    if (!out_dev) {
        if ((rc = ensure_scratch(ctx, std::max<size_t>((size_t)c.width * c.height * 3 * sizeof(float), 256))) != NRRT_OK)
            return rc;
        d_fb = (float*)ctx->scratch;
    }
    if (P.n_owned_pixels) {
        k_resolve<<<(P.n_owned_pixels + 255) / 256, 256, 0, ctx->stream>>>(c, P, nullptr, a->d_sum,
                                                                           (double)a->starts[a->chunks_done], d_fb, packed);
        CK(cudaGetLastError());
    }
    if (out_dev) {
        CK(cudaStreamSynchronize(ctx->stream));
        return NRRT_OK;
    }
    return copy_owned_rows(ctx, o, c.width, c.height, packed, d_fb, out_rgb);
}

int nrrt_accum_sample_map(nrrt_accum* a, uint32_t* out, uint32_t flags) {
    return adaptive_map(a, AMAP_SAMPLES, out, flags, "nrrt_accum_sample_map");
}

int nrrt_accum_error_image(nrrt_accum* a, float* out_rgb, uint32_t flags) {
    return adaptive_map(a, AMAP_ERROR, out_rgb, flags, "nrrt_accum_error_image");
}

int nrrt_accum_save(const nrrt_accum* a, double* sums, uint32_t* samples_done) {
    int rc = accum_check(a, "nrrt_accum_save");
    if (rc != NRRT_OK) return rc;
    nrrt_ctx* ctx = a->ctx;
    if (a->adaptive) {
        ctx->err = "nrrt_accum_save: an adaptive frame's pixels hold different sample counts (nrrt_accum_adaptive_save)";
        return NRRT_ERR_INVALID;
    }
    if ((!sums && a->n_sums) || !samples_done) {
        ctx->err = "nrrt_accum_save: NULL output";
        return NRRT_ERR_INVALID;
    }
    if (a->n_sums) CK(cudaMemcpyAsync(sums, a->d_sum, a->n_sums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *samples_done = a->starts[a->chunks_done];
    return NRRT_OK;
}

int nrrt_accum_restore(nrrt_accum* a, const double* sums, uint32_t samples_done) {
    int rc = accum_check(a, "nrrt_accum_restore");
    if (rc != NRRT_OK) return rc;
    nrrt_ctx* ctx = a->ctx;
    if (a->adaptive) {
        ctx->err = "nrrt_accum_restore: an adaptive frame is restored with nrrt_accum_adaptive_restore";
        return NRRT_ERR_INVALID;
    }
    const auto at = std::find(a->starts.begin(), a->starts.end(), samples_done);
    if (at == a->starts.end()) {
        ctx->err = "nrrt_accum_restore: " + std::to_string(samples_done) + " samples is not a chunk boundary of this frame"
                   " (nrrt_chunk_starts)";
        return NRRT_ERR_INVALID;
    }
    if (!sums && a->n_sums) {
        ctx->err = "nrrt_accum_restore: NULL sums";
        return NRRT_ERR_INVALID;
    }
    if (a->n_sums) CK(cudaMemcpyAsync(a->d_sum, sums, a->n_sums * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    a->chunks_done = (uint32_t)(at - a->starts.begin());
    return NRRT_OK;
}

int nrrt_adaptive_converged(const double S[3], const double Q[3], uint32_t samples, uint32_t chunks,
                            const nrrt_adaptive_opts* adaptive) {
    if (!S || !Q || !adaptive) return 0;
    return adaptive_converged(S, Q, samples, chunks, *adaptive) ? 1 : 0;
}

int nrrt_accum_adaptive_save(const nrrt_accum* a, double* sums, double* sumsq, uint32_t* samples) {
    int rc = accum_check(a, "nrrt_accum_adaptive_save");
    if (rc != NRRT_OK) return rc;
    nrrt_ctx* ctx = a->ctx;
    if (!a->adaptive || (a->n_sums && (!sums || !sumsq || !samples))) {
        ctx->err = a->adaptive ? "nrrt_accum_adaptive_save: NULL output" : "nrrt_accum_adaptive_save: not an adaptive frame";
        return NRRT_ERR_INVALID;
    }
    if (a->n_sums) {
        CK(cudaMemcpyAsync(sums, a->st.S, a->n_sums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(sumsq, a->st.Q, a->n_sums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(samples, a->st.N, a->n_sums / 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return NRRT_OK;
}

int nrrt_accum_adaptive_restore(nrrt_accum* a, const double* sums, const double* sumsq, const uint32_t* samples) {
    const char* who = "nrrt_accum_adaptive_restore";
    int rc = accum_check(a, who);
    if (rc != NRRT_OK) return rc;
    nrrt_ctx* ctx = a->ctx;
    const size_t n = a->n_sums / 3;
    if (!a->adaptive || (n && (!sums || !sumsq || !samples))) {
        ctx->err = std::string(who) + (a->adaptive ? ": NULL input" : ": not an adaptive frame");
        return NRRT_ERR_INVALID;
    }
    // every N a chunk boundary; the frame's boundary is the largest (0: nothing rendered yet, so every N is 0)
    const uint32_t n_chunks = (uint32_t)a->starts.size() - 1;
    std::vector<uint32_t> K(n);
    uint32_t cb = 0;
    for (size_t i = 0; i < n; ++i) {
        const auto at = std::lower_bound(a->starts.begin(), a->starts.end(), samples[i]);
        if (at == a->starts.end() || *at != samples[i]) {
            ctx->err = std::string(who) + ": pixel " + std::to_string(i) + " holds " + std::to_string(samples[i]) +
                       " samples, not a chunk boundary of this frame (nrrt_chunk_starts)";
            return NRRT_ERR_INVALID;
        }
        K[i] = (uint32_t)(at - a->starts.begin());
        cb = std::max(cb, K[i]);
        if (K[i] == 0)  // no samples: nothing may be summed yet, or the first pass would add it in
            for (int ch = 0; ch < 3; ++ch)
                if (sums[3 * i + ch] != 0.0 || sumsq[3 * i + ch] != 0.0) {
                    ctx->err = std::string(who) + ": pixel " + std::to_string(i) + " holds no samples but non-zero sums";
                    return NRRT_ERR_INVALID;
                }
    }
    // pixels below the boundary are retired (they passed the test at their last pass); at the boundary a pixel is
    // active unless it passed it or has every sample.  Active pixels are listed in owned-pixel order, as a pass does.
    const nrrt_camera& c = a->cam;
    const nrrt_render_opts& o = a->opts;
    RenderParams P;
    P.key = make_uint2(0, 0);
    if (const char* why = work_item_params(P, c.width, c.height, c.samples_per_pixel, o.rank, o.world, o.rows_per_block)) {
        ctx->err = std::string(who) + ": " + why;
        return NRRT_ERR_INVALID;
    }
    std::vector<uint32_t> active;
    for (uint32_t po = 0; po < P.n_owned_pixels; ++po) {
        uint32_t x, y, j;
        owned_pixel(c, P, po, x, y, j);
        const size_t pix = (size_t)j * c.width + x;
        const bool conv = adaptive_converged(sums + 3 * pix, sumsq + 3 * pix, samples[pix], K[pix], a->test);
        if (K[pix] < cb && (K[pix] == 0 || !conv)) {
            ctx->err = std::string(who) + ": pixel (" + std::to_string(x) + ", " + std::to_string(y) + ") stopped at " +
                       std::to_string(samples[pix]) + " samples, below the frame's " + std::to_string(a->starts[cb]) +
                       ", without passing the test";
            return NRRT_ERR_INVALID;
        }
        if (K[pix] == cb && (cb == 0 || (cb < n_chunks && !conv))) active.push_back(po);
    }
    if (n) {
        CK(cudaMemcpyAsync(a->st.S, sums, n * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(a->st.Q, sumsq, n * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(a->st.N, samples, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(a->st.K, K.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!active.empty())
        CK(cudaMemcpyAsync(a->d_active[0], active.data(), active.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                           ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    a->cur = 0;
    a->n_active = (uint32_t)active.size();
    a->chunks_done = cb;
    return NRRT_OK;
}

void nrrt_accum_free(nrrt_accum* a) {
    if (!a) return;
    if (a->ctx) {
        cudaSetDevice(a->ctx->device);
        cudaStreamSynchronize(a->ctx->stream);
        accum_release(a);
    } else {
        delete a;
    }
}

// rows of one rank, packed -> their places in the full image (device-output form of nrrt_render_multi)
__global__ void k_place_rows(const float* __restrict__ packed, float* __restrict__ full, uint32_t row_floats, uint32_t n_rows,
                             uint32_t rank, uint32_t world, uint32_t rows_per_block) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n_rows * row_floats) return;
    const uint32_t k = (uint32_t)(i / row_floats), c = (uint32_t)(i - (size_t)k * row_floats);
    const uint32_t b = k / rows_per_block, r = k - b * rows_per_block;  // packed row k = row r of the rank's block b
    full[((size_t)(b * world + rank) * rows_per_block + r) * row_floats + c] = packed[i];
}

int nrrt_render_multi(const int* devices, int n_devices, const nrrt_scene_desc* scene, const nrrt_camera* camera,
                      const nrrt_render_opts* opts_in, float* out_rgb, nrrt_progress_fn progress, void* user,
                      nrrt_render_stats* stats, char* err, size_t err_len) {
    auto fail = [&](const std::string& m, int code) {
        if (err && err_len) std::snprintf(err, err_len, "%s", m.c_str());
        return code;
    };
    if (!devices || n_devices <= 0 || !scene || !camera || !out_rgb) return fail("nrrt_render_multi: bad arguments", NRRT_ERR_INVALID);
    nrrt_render_opts base;
    std::memset(&base, 0, sizeof base);
    if (opts_in) base = *opts_in;
    const bool out_dev = (base.flags & NRRT_RENDER_OUT_DEVICE) != 0;
    if (base.flags & NRRT_RENDER_OUT_PACKED) return fail("nrrt_render_multi: NRRT_RENDER_OUT_PACKED makes no sense here", NRRT_ERR_INVALID);
    const uint32_t world = (uint32_t)n_devices, W = camera->width, H = camera->height;
    const size_t row_floats = (size_t)W * 3;
    struct Rank {
        nrrt_ctx* ctx = nullptr;
        int rc = NRRT_OK;
        std::string msg;
        nrrt_render_stats st{};
        float* d_packed = nullptr;  // device-output form: this rank's packed rows
        uint32_t n_rows = 0;
    };
    std::vector<Rank> ranks(world);
    std::mutex lock;
    std::vector<uint64_t> done(world, 0), total(world, 0);
    struct ProgressCtx {
        std::mutex* lock;
        std::vector<uint64_t>*done, *total;
        uint32_t rank;
        nrrt_progress_fn fn;
        void* user;
    };
    auto on_progress = [](uint64_t d, uint64_t t, void* u) {
        ProgressCtx* p = (ProgressCtx*)u;
        std::lock_guard<std::mutex> g(*p->lock);
        (*p->done)[p->rank] = d, (*p->total)[p->rank] = t;
        uint64_t ds = 0, ts = 0;
        for (size_t i = 0; i < p->done->size(); ++i) ds += (*p->done)[i], ts += (*p->total)[i];
        p->fn(ds, ts, p->user);
    };
    auto work = [&](uint32_t r) {
        Rank& R = ranks[r];
        if ((R.rc = nrrt_create(devices[r], &R.ctx)) != NRRT_OK) {
            R.msg = nrrt_last_error(nullptr);
            return;
        }
        if ((R.rc = nrrt_scene_upload(R.ctx, scene)) != NRRT_OK) {
            R.msg = nrrt_last_error(R.ctx);
            return;
        }
        nrrt_render_opts o = base;
        o.rank = r, o.world = world, o.rows_per_block = world > 1 ? 1 : 0;  // single rows: every device gets the same share of every part of the image
        float* out = out_rgb;
        R.n_rows = owned_rows(H, r, world, world > 1 ? 1 : 8);
        if (out_dev && world > 1) {  // packed rows on this device, gathered on devices[0] below
            if (cudaMalloc((void**)&R.d_packed, std::max<size_t>(1, (size_t)R.n_rows * row_floats * sizeof(float))) != cudaSuccess) {
                R.rc = NRRT_ERR_CUDA, R.msg = "cudaMalloc (packed rows)";
                return;
            }
            o.flags |= NRRT_RENDER_OUT_PACKED;
            out = R.d_packed;
        }
        ProgressCtx pc{&lock, &done, &total, r, progress, user};
        R.rc = nrrt_render(R.ctx, camera, &o, out, progress ? +on_progress : nullptr, &pc, &R.st);
        if (R.rc != NRRT_OK) R.msg = nrrt_last_error(R.ctx);
    };
    std::vector<std::thread> threads;
    for (uint32_t r = 1; r < world; ++r) threads.emplace_back(work, r);
    work(0);
    for (auto& t : threads) t.join();
    int rc = NRRT_OK;
    std::string msg;
    for (uint32_t r = 0; r < world && rc == NRRT_OK; ++r)
        if (ranks[r].rc != NRRT_OK) rc = ranks[r].rc, msg = "device " + std::to_string(devices[r]) + ": " + ranks[r].msg;
    if (rc == NRRT_OK && out_dev && world > 1) {
        // gather on devices[0]: peer copies of the packed rows over NVLink, then one placement kernel per rank
        cudaError_t e = cudaSetDevice(devices[0]);
        float* staging = nullptr;
        size_t max_rows = 0;
        for (auto& R : ranks) max_rows = std::max<size_t>(max_rows, R.n_rows);
        if (e == cudaSuccess) e = cudaMalloc((void**)&staging, std::max<size_t>(1, max_rows * row_floats * sizeof(float)));
        for (uint32_t r = 0; r < world && e == cudaSuccess; ++r) {
            const Rank& R = ranks[r];
            if (!R.n_rows) continue;
            const size_t bytes = (size_t)R.n_rows * row_floats * sizeof(float);
            const float* src = R.d_packed;
            if (r != 0) {
                e = cudaMemcpyPeer(staging, devices[0], R.d_packed, devices[r], bytes);
                src = staging;
            }
            if (e != cudaSuccess) break;
            const size_t n = (size_t)R.n_rows * row_floats;
            k_place_rows<<<(unsigned)((n + 255) / 256), 256>>>(src, out_rgb, (uint32_t)row_floats, R.n_rows, r, world, 1u);
            e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaDeviceSynchronize();
        }
        if (staging) cudaFree(staging);
        if (e != cudaSuccess) rc = NRRT_ERR_CUDA, msg = std::string("gather on device 0: ") + cudaGetErrorString(e);
    }
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        for (auto& R : ranks) {
            stats->paths += R.st.paths, stats->segments += R.st.segments, stats->launches += R.st.launches;
            stats->pixels += R.st.pixels;
            stats->device_ms = std::max(stats->device_ms, R.st.device_ms);
            stats->extend_ms = std::max(stats->extend_ms, R.st.extend_ms);
            stats->extend_launches += R.st.extend_launches;
            stats->mode = R.st.mode;
        }
    }
    for (uint32_t r = 0; r < world; ++r) {
        if (ranks[r].d_packed) {
            cudaSetDevice(devices[r]);
            cudaFree(ranks[r].d_packed);
        }
        nrrt_destroy(ranks[r].ctx);
    }
    if (rc != NRRT_OK) return fail(msg, rc);
    return NRRT_OK;
}

int nrrt_encode_rgb8(nrrt_ctx* ctx, const float* rgb, uint32_t width, uint32_t height, float gamma, uint32_t flags,
                     uint8_t* out_rgb8) {
    if (!ctx) return NRRT_ERR_INVALID;
    if (!rgb || !out_rgb8 || width == 0 || height == 0) {
        ctx->err = "nrrt_encode_rgb8: bad arguments";
        return NRRT_ERR_INVALID;
    }
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)width * height * 3;
    const bool in_dev = (flags & NRRT_RENDER_OUT_DEVICE) != 0;
    // own scratch, kept across calls (the render scratch may hold the very framebuffer being encoded)
    const size_t need = ((n + 255) & ~(size_t)255) + (in_dev ? 0 : n * sizeof(float) + 256);
    if (ctx->enc_bytes < need) {
        if (ctx->enc_buf) {
            CK(cudaStreamSynchronize(ctx->stream));
            CK(cudaFree(ctx->enc_buf));
            ctx->enc_buf = nullptr, ctx->enc_bytes = 0;
        }
        CK(cudaMalloc(&ctx->enc_buf, need));
        ctx->enc_bytes = need;
    }
    uint8_t* d_out = (uint8_t*)ctx->enc_buf;
    const float* d_in = rgb;
    if (!in_dev) {
        float* staged = (float*)((char*)ctx->enc_buf + ((n + 255) & ~(size_t)255));
        CK(cudaMemcpyAsync(staged, rgb, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        d_in = staged;
    }
    k_encode_rgb8<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_in, n, gamma, d_out);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out_rgb8, d_out, n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return NRRT_OK;
}

// struct sizes, so bindings can verify their mirror of the header
size_t nrrt_abi_sizeof(int which) {
    switch (which) {
        case 0: return sizeof(nrrt_object);
        case 1: return sizeof(nrrt_material);
        case 2: return sizeof(nrrt_texture);
        case 3: return sizeof(nrrt_image);
        case 4: return sizeof(nrrt_graph_desc);
        case 5: return sizeof(nrrt_camera_config);
        case 6: return sizeof(nrrt_camera);
        case 7: return sizeof(nrrt_node);
        case 8: return sizeof(nrrt_box);
        case 9: return sizeof(nrrt_xform);
        case 10: return sizeof(nrrt_instance);
        case 11: return sizeof(nrrt_scene_desc);
        case 12: return sizeof(nrrt_hit);
        case 13: return sizeof(nrrt_trace_stats);
        case 14: return sizeof(nrrt_render_opts);
        case 15: return sizeof(nrrt_render_stats);
        case 16: return sizeof(nrrt_camera_file);
        case 17: return sizeof(nrrt_wnode);
        case 18: return sizeof(nrrt_hit_compact);
        case 19: return sizeof(nrrt_adaptive_opts);
        default: return 0;
    }
}

}  // extern "C"
