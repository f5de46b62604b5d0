// rrtb_render.cu -- the render megakernels and the parity-test hooks (sm_100a).
//
// Replaces render_init + cuda_render (rrt.cu:81-122) and ray_color (rrt.cu:42-79).  k_render below is the
// one-path-per-lane kernel of the flat scan and RRTB_SCHED_SIMPLE; the LBVH default is the pool scheduler of
// rrtb_render_pool.cuh.  Both kernels and the hooks are written once over the path policy of rrtb_path.cuh and
// instantiated for the float and the double integrator; both kernels shade a segment with hit_step / miss_fixed and
// map a work item to its pixel and sample with local_pixel / global_sample below.
//
// Scheduling.  The reference runs one thread per PIXEL, so a warp lives until its slowest pixel has
// finished all spp samples of up to max_depth bounces.  Here the kernel is PERSISTENT: the grid is
// (resident blocks per SM) x 148 SMs and every lane loops
//
//      fetch work item  ->  [ generate primary ray -> (trace one segment -> shade)* ]* -> flush
//
// A work item is (pixel, chunk of <= CHUNK samples).  Items are handed out by one warp-aggregated
// atomicAdd on a global queue head (ballot + popc, one atomic per refill).  A lane that terminates a
// path regenerates the next sample of its own item in place, so all 32 lanes trace a segment on every
// trip round the loop until the queue drains (Aila & Laine 2009 persistent threads + in-warp path
// regeneration).  Items of 32 consecutive indices are the 8x4 pixels of one image tile, so a freshly
// filled warp starts with coherent primary rays.
//
// Determinism.  All randomness comes from Philox4x32-10 keyed by (pixel, sample, bounce); a lane sums
// the radiance of its chunk in 2^40 fixed point and flushes with 64-bit integer atomics.  Integer
// addition is associative, so the image is bit-identical for any grid size, any scheduling, tile- or
// sample-sharding across GPUs and any reduction order (NCCL or peer atomics).
#include "rrtb_internal.h"
#include "rrtb_path.cuh"

#include <stdio.h>
#include <stdlib.h>

namespace rrtb {

static constexpr int RENDER_TPB = 256;
static constexpr int CHUNK = 16; // samples per work item
#ifndef RRTB_NODE_UNROLL
#define RRTB_NODE_UNROLL 2
#endif
static constexpr int NODE_UNROLL = RRTB_NODE_UNROLL; // wide-node visits between two continue-votes of the pool scheduler

struct RenderArgs {
    DeviceScene scene;
    DeviceCamera cam;
    int W, H, spp, max_depth;
    float clamp; // per-sample radiance clamp of the whole render, fixed_clamp(spp)
    uint2 key;
    int rank, world, shard_mode;
    int tiles_x, tiles_y;
    int n_local_tiles;   // tiles owned by this rank
    int n_local_samples; // samples owned by this rank
    int n_chunks;        // ceil(n_local_samples / CHUNK)
    unsigned long long n_items; // n_local_tiles * n_chunks * 32
    unsigned long long *accum;  // 3*W*H fixed-point sums
    int th_fetch, th_shade, th_leaf; // pool-scheduler thresholds (lanes)
    int step_iters, th_node;         // max node visits per scheduling round / lanes needed to continue
    unsigned long long *queue;  // [0] queue head, [1] rays, [2] box tests, [3] sphere, [4] msphere, [5] triangle tests, [6] hits
    // LIGHTS kernels only (appended, so the fields above keep their parameter offsets)
    int background;             // != 0: a segment that leaves the scene adds throughput x bg instead of the sky
    float bg[3];
};

// ---- the rules of a work item and of a path segment, shared by the lane kernel and the pool scheduler ----------------
// The pool passes its slot fields to the reference parameters, so that each is read from shared memory only where used.

// The pixel (i, j) of pixel-in-tile `pit` of 8x4-pixel tile `tile` (row-major, tiles_x per row).
__device__ __forceinline__ void tile_pixel(int tile, int tiles_x, unsigned pit, int &i, int &j)
{
    int ty = (int)__fdividef((float)tile, (float)tiles_x); // float estimate, off by <= 1 below 2^28 pixels ...
    int tx = tile - ty * tiles_x;
    if (tx < 0) { // ... corrected exactly in integers
        --ty;
        tx += tiles_x;
    }
    else if (tx >= tiles_x) {
        ++ty;
        tx -= tiles_x;
    }
    i = tx * 8 + (int)(pit & 7u);
    j = ty * 4 + (int)(pit >> 3);
}

// The pixel of pixel-in-tile `pit` of this rank's local tile `ltile`; false for a padding pixel of an edge tile.
__device__ __forceinline__ bool local_pixel(const RenderArgs &a, int ltile, unsigned pit, int &i, int &j)
{
    tile_pixel(a.shard_mode == RRTB_SHARD_TILES ? ltile * a.world + a.rank : ltile, a.tiles_x, pit, i, j);
    return i < a.W && j < a.H;
}

// The sample of this rank's local sample `ls`, the key of its Philox streams.
__device__ __forceinline__ int global_sample(const RenderArgs &a, int ls)
{
    return a.shard_mode == RRTB_SHARD_SAMPLES ? ls * a.world + a.rank : ls;
}

// A segment that leaves the scene adds background x throughput (LIGHTS, a scene with a background), else sky x
// throughput (rrt.cu:68-75); the sky reads only the ray's direction.
template <class P, bool LIGHTS>
__device__ __forceinline__ ulonglong3 miss_fixed(const RenderArgs &a, const typename P::RayT &ray, const typename P::real &tr,
                                                 const typename P::real &tg, const typename P::real &tb)
{
    ulonglong3 f;
    if (LIGHTS && a.background) P::const_fixed(tr, tg, tb, a.bg[0], a.bg[1], a.bg[2], a.clamp, f.x, f.y, f.z);
    else P::sky_fixed(ray, tr, tg, tb, a.clamp, f.x, f.y, f.z);
    return f;
}

// A segment that hit something (rrt.cu:50-63): hit record, Philox block (pixel, sample, 2 + bounce), scatter.  True:
// the path goes on, with `ray` and the throughput updated.  False: it ends; an emitter (LIGHTS) hands its last term,
// throughput x Le, to `emit`, called behind the material test alone so that the pool's atomics need no test of their
// own.  A scattered path ends here when its next segment would exceed max_depth (rrt.cu:78);
// such a segment would add nothing, so ending the path one segment later gives the same image.
template <class P, bool MTRI, bool LIGHTS, class Emit>
__device__ __forceinline__ bool hit_step(const RenderArgs &a, const float4 *__restrict__ leaves, const LeafAux info,
                                         typename P::RayT &ray, const typename P::HitT &h, const int &pixel, const int &sample,
                                         int bounce, typename P::real &tr, typename P::real &tg, typename P::real &tb,
                                         const Emit &emit)
{
    const typename P::RecT rec = P::template record<MTRI>(leaves, info, ray, h);
    const uint4 rnd = philox4x32_10(make_uint4((uint32_t)pixel, (uint32_t)sample, 2u + (uint32_t)bounce, 0u), a.key);
    const float4 m = __ldg(&a.scene.materials[rec.mat]);
    const int mtype = __ldg(&a.scene.material_type[rec.mat]);
    typename P::real dx, dy, dz, ar, ag, ab;
    const bool go_on = P::template bounce<LIGHTS>(mtype, m, ray, rec, rnd, dx, dy, dz, ar, ag, ab) && bounce + 1 < a.max_depth;
    if (go_on) {
        ray.ox = rec.px; ray.oy = rec.py; ray.oz = rec.pz;
        ray.dx = dx; ray.dy = dy; ray.dz = dz;
        tr = P::mul(tr, ar); tg = P::mul(tg, ag); tb = P::mul(tb, ab);
    }
    else if constexpr (LIGHTS) { // (if constexpr: the other instantiations keep their code exactly)
        if (mtype == RRTB_DIFFUSE_LIGHT) {
            ulonglong3 f;
            P::const_fixed(tr, tg, tb, m.x, m.y, m.z, a.clamp, f.x, f.y, f.z);
            emit(f);
        }
    }
    return go_on;
}

// Adds a fixed-point triple to a pixel's sums (64-bit integer atomics: the order of arrival does not matter).
__device__ __forceinline__ void accumulate(const RenderArgs &a, int pixel, ulonglong3 f)
{
    unsigned long long *dst = a.accum + 3ull * (unsigned long long)pixel;
    atomicAdd(dst + 0, f.x);
    atomicAdd(dst + 1, f.y);
    atomicAdd(dst + 2, f.z);
}

// Counting build: the warp's sums of {rays, box, sphere, msphere, triangle tests, hits} into queue[1..6].
__device__ __forceinline__ void flush_counters(const RenderArgs &a, unsigned long long rays, const TravCounters &tc,
                                               unsigned long long hits)
{
    unsigned long long v[6] = {rays, tc.box, tc.sph, tc.msph, tc.tri, hits};
    for (int k = 0; k < 6; ++k) {
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        if ((threadIdx.x & 31u) == 0 && v[k]) atomicAdd(a.queue + 1 + k, v[k]);
    }
}

// LIGHTS: the scene has emitters (RRTB_DIFFUSE_LIGHT) or a background; the other instantiations compile neither in
template <class P, bool USE_BVH, bool COUNT_RAYS, bool LIGHTS = false>
__global__ void __launch_bounds__(RENDER_TPB, 2) k_render(const RenderArgs a)
{
    typedef typename P::real real;
    const unsigned lane = threadIdx.x & 31u;
    const DeviceScene &s = a.scene;
    const float4 *__restrict__ leaves = USE_BVH ? s.leaves : s.flat_leaves;
    const LeafAux info = USE_BVH ? LeafAux{s.leaf_info, s.leaf_ext} : LeafAux{s.flat_info, s.flat_ext};

    // lane state
    int pixel = -1, ls = 0, ls_end = 0; // current item: pixel, local sample cursor, end
    ulonglong3 acc = make_ulonglong3(0ull, 0ull, 0ull); // the item's radiance so far, fixed point
    typename P::RayT ray;
    real thr_r = 1, thr_g = 1, thr_b = 1;
    int bounce = 0;
    bool in_path = false;
    bool done = false;
    unsigned long long rays = 0, hits = 0;
    TravCounters tc = {0ull, 0ull, 0ull, 0ull};

    while (true) {
        // ---- refill: lanes without a current item pull the next items off the queue -------------------
        bool need = !done && pixel < 0;
        unsigned need_mask = __ballot_sync(0xffffffffu, need);
        if (need_mask) {
            unsigned long long base = 0;
            const int leader = __ffs(need_mask) - 1;
            if ((int)lane == leader) base = atomicAdd(a.queue, (unsigned long long)__popc(need_mask));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (need) {
                unsigned long long item = base + __popc(need_mask & ((1u << lane) - 1u));
                if (item >= a.n_items) {
                    done = true;
                }
                else {
                    // item = (local_tile * n_chunks + chunk) * 32 + pixel_in_tile
                    unsigned pit = (unsigned)(item & 31ull);
                    unsigned long long tile_chunk = item >> 5;
                    int chunk = (int)(tile_chunk % (unsigned long long)a.n_chunks);
                    int ltile = (int)(tile_chunk / (unsigned long long)a.n_chunks);
                    int i, j;
                    if (local_pixel(a, ltile, pit, i, j)) {
                        pixel = j * a.W + i;
                        ls = chunk * CHUNK;
                        ls_end = min(ls + CHUNK, a.n_local_samples);
                        in_path = false;
                    } // else: padding pixel of an edge tile; stays idle this round, refills next round
                }
            }
        }
        if (__all_sync(0xffffffffu, done)) break;

        if (pixel >= 0) {
            const int sample = global_sample(a, ls);
            if (!in_path) { // ---- generate: rrt.cu:112-114 + camera.h:31-38
                ray = P::camera(a.cam, a.W, a.H, pixel % a.W, pixel / a.W, sample, a.key);
                thr_r = thr_g = thr_b = 1;
                bounce = 0;
                in_path = true;
            }
            // ---- extend: one closest-hit query (rrt.cu:49)
            const real t_min = (real)0.001;
            typename P::HitT h = USE_BVH ? closest_bvh<P, COUNT_RAYS>(s, ray, t_min, tc) : closest_scan<P, COUNT_RAYS>(s, ray, t_min, tc);
            if (COUNT_RAYS) {
                ++rays;
                if (h.ref >= 0) ++hits;
            }
            // ---- shade: rrt.cu:50-76
            const auto add = [&](ulonglong3 f) { acc.x += f.x; acc.y += f.y; acc.z += f.z; };
            if (h.ref < 0) add(miss_fixed<P, LIGHTS>(a, ray, thr_r, thr_g, thr_b));
            else if (hit_step<P, true, LIGHTS>(a, leaves, info, ray, h, pixel, sample, bounce, thr_r, thr_g, thr_b, add)) {
                ++bounce;
                continue; // the path goes on
            }
            in_path = false;
            if (++ls >= ls_end) { // ---- flush the chunk
                accumulate(a, pixel, acc);
                acc = make_ulonglong3(0ull, 0ull, 0ull);
                pixel = -1;
            }
        }
    }
    if (COUNT_RAYS) flush_counters(a, rays, tc, hits);
}

// ---- first-hit AOVs (rrtb_render_aov) -----------------------------------------------------------------------------
// The primary segment of every sample of a pixel: camera ray, one closest-hit query, and on a hit the clamped albedo,
// the face-forwarded normal of the hit record and the distance t |d|.  A lane owns one pixel and runs its samples in
// order, summing in double (a miss leaves the sums as they are), so the means depend on neither the grid nor the tree.
struct AovArgs {
    DeviceScene scene;
    DeviceCamera cam;
    int W, H, spp;
    uint2 key;
    int rank, world, tiles_x;
    int n_local_tiles;         // tiles owned by this rank (RRTB_SHARD_TILES)
    float *out;                // planar: albedo 3*W*H, normal 3*W*H, depth W*H, coverage W*H
    unsigned long long *queue; // [0] tile queue head, [1..6] the counters of RenderArgs::queue
};

// persistent: each warp draws one 8x4-pixel tile at a time off the queue, lane = pixel in tile
template <class P, bool USE_BVH, bool COUNT_RAYS>
__global__ void __launch_bounds__(RENDER_TPB, 2) k_render_aov(const AovArgs a)
{
    typedef typename P::real real;
    const unsigned lane = threadIdx.x & 31u;
    const DeviceScene &s = a.scene;
    const float4 *__restrict__ leaves = USE_BVH ? s.leaves : s.flat_leaves;
    const LeafAux info = USE_BVH ? LeafAux{s.leaf_info, s.leaf_ext} : LeafAux{s.flat_info, s.flat_ext};
    const size_t n = (size_t)a.W * a.H;
    unsigned long long rays = 0, hits = 0;
    TravCounters tc = {0ull, 0ull, 0ull, 0ull};

    while (true) {
        unsigned long long ltile = 0;
        if (lane == 0) ltile = atomicAdd(a.queue, 1ull);
        ltile = __shfl_sync(0xffffffffu, ltile, 0);
        if (ltile >= (unsigned long long)a.n_local_tiles) break;
        int i, j;
        tile_pixel((int)ltile * a.world + a.rank, a.tiles_x, lane, i, j);
        if (i >= a.W || j >= a.H) continue; // padding pixel of an edge tile
        double al[3] = {0.0, 0.0, 0.0}, nm[3] = {0.0, 0.0, 0.0}, dist = 0.0;
        int n_hit = 0;
        for (int smp = 0; smp < a.spp; ++smp) {
            const typename P::RayT ray = P::camera(a.cam, a.W, a.H, i, j, smp, a.key);
            const real t_min = (real)0.001;
            const typename P::HitT h = USE_BVH ? closest_bvh<P, COUNT_RAYS>(s, ray, t_min, tc) : closest_scan<P, COUNT_RAYS>(s, ray, t_min, tc);
            if (COUNT_RAYS) {
                ++rays;
                if (h.ref >= 0) ++hits;
            }
            if (h.ref < 0) continue;
            const typename P::RecT rec = P::template record<true>(leaves, info, ray, h);
            real ar, ag, ab;
            P::albedo(__ldg(&s.material_type[rec.mat]), __ldg(&s.materials[rec.mat]), ar, ag, ab);
            al[0] = __dadd_rn(al[0], (double)ar);
            al[1] = __dadd_rn(al[1], (double)ag);
            al[2] = __dadd_rn(al[2], (double)ab);
            nm[0] = __dadd_rn(nm[0], (double)rec.nx);
            nm[1] = __dadd_rn(nm[1], (double)rec.ny);
            nm[2] = __dadd_rn(nm[2], (double)rec.nz);
            dist = __dadd_rn(dist, (double)P::distance(ray, h.t));
            ++n_hit;
        }
        // each mean: one correctly rounded division, one rounding to float
        const double spp = (double)a.spp;
        const size_t p = (size_t)j * a.W + i;
        for (int k = 0; k < 3; ++k) {
            a.out[3 * p + k] = __double2float_rn(__ddiv_rn(al[k], spp));
            a.out[3 * n + 3 * p + k] = __double2float_rn(__ddiv_rn(nm[k], spp));
        }
        a.out[6 * n + p] = n_hit ? __double2float_rn(__ddiv_rn(dist, (double)n_hit)) : 0.0f;
        a.out[7 * n + p] = __double2float_rn(__ddiv_rn((double)n_hit, spp));
    }
    if (COUNT_RAYS) { // the warp's sums of {rays, box, sphere, msphere, triangle tests, hits} into queue[1..6], as flush_counters
        unsigned long long v[6] = {rays, tc.box, tc.sph, tc.msph, tc.tri, hits};
        for (int k = 0; k < 6; ++k) {
            for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
            if (lane == 0 && v[k]) atomicAdd(a.queue + 1 + k, v[k]);
        }
    }
}

} // namespace rrtb
#include "rrtb_render_pool.cuh"
namespace rrtb {

// fixed point -> float or double; the float is one rounding of the double product (exact below 2^53)
template <typename T>
__global__ void k_resolve(const unsigned long long *__restrict__ acc, T *__restrict__ out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = (T)((double)acc[i] * 9.094947017729282e-13); // 2^-40
}

// Multi-GPU epilogue of a tile shard (SURVEY 8e): one warp per OWNED 8x4-pixel tile converts its 32 accumulators and
// stores them as 3 floats (or doubles) straight into the owner's frame -- `out` is rank 0's buffer, for ranks > 0 a
// peer mapping over NVLink.  Tiles are disjoint, so the frame needs neither a zero-fill nor a reduction:
// 12 B/pixel/GPU cross the link instead of a 24 B/pixel full-frame integer reduce.
template <typename T>
__global__ void __launch_bounds__(256) k_resolve_tiles(const unsigned long long *__restrict__ acc, T *out, int W, int H,
                                                        int tiles_x, int n_tiles, int rank, int world)
{
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (int tile = rank + warp * world; tile < n_tiles; tile += n_warps * world) {
        int i, j;
        tile_pixel(tile, tiles_x, lane, i, j);
        if (i < W && j < H) {
            const size_t k = 3 * ((size_t)j * W + i);
            out[k + 0] = (T)((double)acc[k + 0] * 9.094947017729282e-13); // 2^-40; float: one rounding, as k_resolve
            out[k + 1] = (T)((double)acc[k + 1] * 9.094947017729282e-13);
            out[k + 2] = (T)((double)acc[k + 2] * 9.094947017729282e-13);
        }
    }
}

// Multi-GPU epilogue of a sample shard: the partial sums are ADDED into the owner's 64-bit accumulator (integer
// atomics, over NVLink for ranks > 0): associative, so the image does not depend on the arrival order.
__global__ void k_accumulate_atomic(unsigned long long *dst, const unsigned long long *__restrict__ src, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const unsigned long long v = src[i];
        if (v) atomicAdd(dst + i, v);
    }
}

__global__ void k_accumulate(unsigned long long *__restrict__ dst, const unsigned long long *__restrict__ src, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) dst[i] += src[i];
}

// ---- test-hook kernels: they call the SAME device functions the render kernels inline -----------------
template <class P>
__global__ void k_trace(const DeviceScene s, const typename P::real *__restrict__ rays7, int n, typename P::real t_min, int mode,
                        int *__restrict__ id, typename P::real *__restrict__ t, typename P::real *__restrict__ rec7)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const typename P::real *q = rays7 + 7 * (size_t)i;
    typename P::RayT r;
    r.ox = q[0]; r.oy = q[1]; r.oz = q[2]; r.dx = q[3]; r.dy = q[4]; r.dz = q[5]; r.tm = q[6];
    TravCounters tc;
    typename P::HitT h = mode ? closest_bvh<P, false>(s, r, t_min, tc) : closest_scan<P, false>(s, r, t_min, tc);
    if (h.ref < 0) {
        id[i] = -1;
        t[i] = -1;
        if (rec7)
            for (int k = 0; k < 7; ++k) rec7[7 * (size_t)i + k] = 0;
        return;
    }
    typename P::RecT rec = P::template record<true>(mode ? s.leaves : s.flat_leaves,
                                                    mode ? LeafAux{s.leaf_info, s.leaf_ext} : LeafAux{s.flat_info, s.flat_ext}, r, h);
    id[i] = rec.obj;
    t[i] = h.t;
    if (rec7) {
        typename P::real *o = rec7 + 7 * (size_t)i;
        o[0] = rec.px; o[1] = rec.py; o[2] = rec.pz; o[3] = rec.nx; o[4] = rec.ny; o[5] = rec.nz;
        o[6] = rec.front ? 1 : 0;
    }
}

template <class P>
__global__ void k_camera_rays(const DeviceCamera cam, int W, int H, uint2 key, const int *__restrict__ pix, int n,
                              int sample, typename P::real *__restrict__ rays7)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    typename P::RayT r = P::camera(cam, W, H, pix[i] % W, pix[i] / W, sample, key);
    typename P::real *o = rays7 + 7 * (size_t)i;
    o[0] = r.ox; o[1] = r.oy; o[2] = r.oz; o[3] = r.dx; o[4] = r.dy; o[5] = r.dz; o[6] = r.tm;
}

__global__ void k_philox(const uint32_t *__restrict__ ctr, int n, uint2 key, uint32_t *__restrict__ out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 c = make_uint4(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]);
    uint4 o = philox4x32_10(c, key);
    out[4 * i] = o.x; out[4 * i + 1] = o.y; out[4 * i + 2] = o.z; out[4 * i + 3] = o.w;
}

template <class P>
__global__ void k_scatter_test(const DeviceScene s, const typename P::real *__restrict__ in16, const uint32_t *__restrict__ rnd4,
                               int n, typename P::real *__restrict__ out8)
{
    typedef typename P::real real;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const real *in = in16 + 16 * (size_t)i;
    typename P::RayT r;
    r.ox = in[0]; r.oy = in[1]; r.oz = in[2]; r.dx = in[3]; r.dy = in[4]; r.dz = in[5]; r.tm = in[6];
    typename P::RecT rec;
    rec.px = in[7]; rec.py = in[8]; rec.pz = in[9];
    rec.nx = in[10]; rec.ny = in[11]; rec.nz = in[12];
    rec.front = in[13] != 0;
    rec.mat = (int)in[14];
    rec.obj = 0;
    uint4 rnd = make_uint4(rnd4[4 * i], rnd4[4 * i + 1], rnd4[4 * i + 2], rnd4[4 * i + 3]);
    real dx, dy, dz, ar, ag, ab;
    bool ok = P::template bounce<true>(__ldg(&s.material_type[rec.mat]), __ldg(&s.materials[rec.mat]), r, rec, rnd, dx, dy, dz, ar, ag, ab);
    real *o = out8 + 8 * (size_t)i;
    o[0] = dx; o[1] = dy; o[2] = dz; o[3] = ar; o[4] = ag; o[5] = ab; o[6] = ok ? 1 : 0; o[7] = 0;
}

// ---- issue-rate probe: the measured denominator of the FP32-issue roofline (SURVEY 8d) -----------------
// MIX = false: 8 independent FFMA chains per thread (fma pipe only).
// MIX = true : FFMA + FMNMX interleaved (fma pipe + alu pipe), the instruction mix of a slab test.
template <bool MIX>
__global__ void __launch_bounds__(256) k_probe(float *out, int iters, float seed)
{
    float a0 = seed + threadIdx.x, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f,
          a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.999999f, c = 1e-7f;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
            a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
            if (MIX) {
                a0 = fminf(a0, a4); a1 = fmaxf(a1, a5); a2 = fminf(a2, a6); a3 = fmaxf(a3, a7);
                a4 = fmaxf(a4, a1); a5 = fminf(a5, a2); a6 = fmaxf(a6, a3); a7 = fminf(a7, a0);
            }
        }
    }
    float r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (r == 123.456f) out[0] = r; // never true; keeps the chains alive
}

int launch_probe(rrtb_ctx *ctx, int mix, double *lane_instr_per_s)
{
    const int iters = 4096, blocks = ctx->sm_count * 8;
    float *d_out = (float *)ctx->d_counters;
    float ms = 0.f;
    for (int rep = 0; rep < 3; ++rep) { // last repetition is the measurement
        RRTB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        if (mix) k_probe<true><<<blocks, 256, 0, ctx->stream>>>(d_out, iters, 1.0f);
        else k_probe<false><<<blocks, 256, 0, ctx->stream>>>(d_out, iters, 1.0f);
        RRTB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        RRTB_CUDA(ctx, cudaGetLastError());
        RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        RRTB_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    }
    const double per_thread = (double)iters * 8.0 * (mix ? 16.0 : 8.0);
    *lane_instr_per_s = per_thread * 256.0 * blocks / (ms * 1e-3);
    return RRTB_OK;
}

// ---- host launchers ---------------------------------------------------------------------------------------
DeviceScene device_scene(const rrtb_ctx *ctx)
{
    DeviceScene s;
    s.wnodes = ctx->d_wnodes;
    s.motion = ctx->motion ? 1 : 0;
    s.shutter_open = ctx->cam.time0;
    s.shutter_inv = ctx->motion ? 1.0f / (ctx->cam.time1 - ctx->cam.time0) : 0.f;
    s.leaves = ctx->d_leaves;
    s.leaf_info = ctx->d_leaf_info;
    s.flat_leaves = ctx->d_prim;
    s.flat_info = ctx->d_prim_info;
    s.leaf_ext = ctx->d_leaf_ext;
    s.flat_ext = ctx->d_prim_ext;
    s.materials = ctx->d_materials;
    s.material_type = ctx->d_material_type;
    s.n_prims = ctx->n_prims;
    s.n_spheres = ctx->n_spheres;
    s.n_mspheres = ctx->n_mspheres;
    s.n_triangles = ctx->n_triangles;
    s.n_mtriangles = ctx->n_mtriangles;
    s.use_bvh = ctx->use_bvh;
    return s;
}

DeviceCamera device_camera(const rrtb_camera &c, int W, int H)
{
    DeviceCamera d;
    d.inv_w1 = 1.0f / (float)(W - 1);
    d.inv_h1 = 1.0f / (float)(H - 1);
    for (int k = 0; k < 3; ++k) {
        d.origin[k] = c.origin[k];
        d.llc[k] = c.lower_left_corner[k];
        d.horizontal[k] = c.horizontal[k];
        d.vertical[k] = c.vertical[k];
        d.u[k] = c.u[k];
        d.v[k] = c.v[k];
        d.w[k] = c.w[k];
    }
    d.lens_radius = c.lens_radius;
    d.time0 = c.time0;
    d.time1 = c.time1;
    return d;
}

// The 8x4-pixel tiles of a frame and the share of rank `rank` of `world`: under RRTB_SHARD_TILES the tiles
// t with t % world == rank and every sample, under RRTB_SHARD_SAMPLES every tile and the samples s with s % world == rank.
struct ShardGeometry {
    int world, rank, tiles_x, tiles_y, n_tiles, n_local_tiles, n_local_samples;
};

static ShardGeometry shard_geometry(const rrtb_render_params *p)
{
    ShardGeometry g;
    g.world = p->world < 1 ? 1 : p->world;
    g.rank = p->world < 1 ? 0 : p->rank;
    g.tiles_x = (p->width + 7) / 8;
    g.tiles_y = (p->height + 3) / 4;
    g.n_tiles = g.tiles_x * g.tiles_y;
    const bool tiles = p->shard_mode == RRTB_SHARD_TILES;
    g.n_local_tiles = tiles ? max((g.n_tiles - g.rank + g.world - 1) / g.world, 0) : g.n_tiles;
    g.n_local_samples = tiles ? p->spp : max((p->spp - g.rank + g.world - 1) / g.world, 0);
    return g;
}

// blocks of 256 threads for a grid-stride loop over n elements: one element per thread, at most 8 blocks per SM
static int grid_size(const rrtb_ctx *ctx, size_t n)
{
    const size_t blocks = (n + 255) / 256, cap = (size_t)ctx->sm_count * 8;
    return (int)(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
}

// the lane kernel: persistent, one wave, a multiple of the SM count
template <class P, bool USE_BVH, bool LIGHTS = false>
static int launch_lane(rrtb_ctx *ctx, const RenderArgs &args, bool cnt, int *blocks_out)
{
    auto kernel = cnt ? k_render<P, USE_BVH, true, LIGHTS> : k_render<P, USE_BVH, false, LIGHTS>;
    int per_sm = 0;
    RRTB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, RENDER_TPB, 0));
    if (per_sm < 1) per_sm = 1;
    unsigned long long want = (args.n_items + RENDER_TPB - 1) / RENDER_TPB;
    int blocks = ctx->sm_count * per_sm;
    if ((unsigned long long)blocks > want) blocks = (int)(want ? want : 1);
    kernel<<<blocks, RENDER_TPB, 0, ctx->stream>>>(args);
    *blocks_out = blocks;
    return RRTB_OK;
}

template <class P, bool MTRI, bool MOTION, bool LIGHTS = false>
static int launch_pool(rrtb_ctx *ctx, const RenderArgs &args, bool cnt, int *blocks_out)
{
    auto kernel = cnt ? k_render_pool<true, NODE_UNROLL, MTRI, P, MOTION, LIGHTS> : k_render_pool<false, NODE_UNROLL, MTRI, P, MOTION, LIGHTS>;
    constexpr int POOL = P::POOL;
    const int smem = (int)(sizeof(WarpPoolT<typename P::real, POOL>) * POOL_WARPS);
    RRTB_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    RRTB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, RENDER_TPB, smem));
    if (per_sm < 1) per_sm = 1;
    // persistent: one wave; every warp needs at least a pool's worth of paths to be worth launching
    unsigned long long want = (args.n_items + (unsigned long long)POOL * POOL_WARPS - 1) / ((unsigned long long)POOL * POOL_WARPS);
    int blocks = ctx->sm_count * per_sm;
    if ((unsigned long long)blocks > want) blocks = (int)(want ? want : 1);
    kernel<<<blocks, RENDER_TPB, smem, ctx->stream>>>(args);
    *blocks_out = blocks;
    return RRTB_OK;
}

int launch_render(rrtb_ctx *ctx, const rrtb_render_params *p, uint64_t *d_accum, rrtb_stats *stats, bool defer)
{
    const ShardGeometry g = shard_geometry(p);
    RenderArgs a;
    a.scene = device_scene(ctx);
    a.cam = device_camera(ctx->cam, p->width, p->height);
    a.W = p->width;
    a.H = p->height;
    a.spp = p->spp;
    a.clamp = fixed_clamp(p->spp); // the total spp, not the shard's: every shard clamps alike
    a.max_depth = p->max_depth;
    a.key = make_uint2((uint32_t)p->seed, (uint32_t)(p->seed >> 32));
    a.world = g.world;
    a.rank = g.rank;
    a.shard_mode = p->shard_mode;
    a.tiles_x = g.tiles_x;
    a.tiles_y = g.tiles_y;
    a.n_local_tiles = g.n_local_tiles;
    a.n_local_samples = g.n_local_samples;
    a.n_chunks = (a.n_local_samples + CHUNK - 1) / CHUNK;
    const bool use_pool = ctx->use_bvh != 0 && p->scheduler != RRTB_SCHED_SIMPLE;
    // the lane kernel hands out chunks of CHUNK samples of a pixel, the pool scheduler single camera paths:
    // (tile, chunk or sample, pixel in tile)
    a.n_items = (unsigned long long)a.n_local_tiles * (unsigned long long)(use_pool ? a.n_local_samples : a.n_chunks) * 32ull;
    a.accum = (unsigned long long *)d_accum;
    a.th_fetch = 16;
    a.th_shade = 32;
    a.th_leaf = 8;
    a.step_iters = 8;
    a.th_node = 12;
#ifdef RRTB_TUNING // tuning build only (make tune): scheduler thresholds from the environment, clamped to what the kernel assumes
    auto knob = [](const char *name, int dflt, int lo, int hi) {
        const char *e = getenv(name);
        if (!e) return dflt;
        const int v = atoi(e);
        return v < lo ? lo : (v > hi ? hi : v);
    };
    a.step_iters = knob("RRTB_STEP_ITERS", a.step_iters, 1, 1 << 20);
    a.th_node = knob("RRTB_TH_NODE", a.th_node, 1, 32);
    a.th_fetch = knob("RRTB_TH_FETCH", a.th_fetch, 1, 32);
    a.th_shade = knob("RRTB_TH_SHADE", a.th_shade, 1, 32);
    a.th_leaf = knob("RRTB_TH_LEAF", a.th_leaf, 1, 32);
#endif
    a.queue = ctx->d_counters;
    a.background = ctx->background ? 1 : 0;
    for (int k = 0; k < 3; ++k) a.bg[k] = ctx->bg[k];

    RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_counters, 0, 8 * sizeof(unsigned long long), ctx->stream));
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int blocks = 0;
    int launches = 0;
    if (a.n_items > 0 && a.max_depth > 0) { // max_depth 0: the bounce loop never runs (rrt.cu:47), the image is black
        typedef int (*Launcher)(rrtb_ctx *, const RenderArgs &, bool, int *);
        // the lane kernel, [precision][use_bvh]: flat scan or LBVH
        static const Launcher lane[2][2] = {{launch_lane<PathF32, false>, launch_lane<PathF32, true>},
                                            {launch_lane<PathF64, false>, launch_lane<PathF64, true>}};
        // the pool scheduler, [policy][motion nodes]; MTRI compiles the moving-triangle cases in: the float kernel has
        // them only for scenes with moving triangles (SURVEY 8f4), the double kernel always
        static const Launcher pool[3][2] = {{launch_pool<PathF32, false, false>, launch_pool<PathF32, false, true>},
                                            {launch_pool<PathF32, true, false>, launch_pool<PathF32, true, true>},
                                            {launch_pool<PathF64, true, false>, launch_pool<PathF64, true, true>}};
        // scenes with emitters or a background (ctx->lights): the LIGHTS kernels, [precision][...] as above; the float pool
        // kernel compiles the moving-triangle cases in, as the double one does
        static const Launcher lane_lit[2][2] = {{launch_lane<PathF32, false, true>, launch_lane<PathF32, true, true>},
                                                {launch_lane<PathF64, false, true>, launch_lane<PathF64, true, true>}};
        static const Launcher pool_lit[2][2] = {{launch_pool<PathF32, true, false, true>, launch_pool<PathF32, true, true, true>},
                                                {launch_pool<PathF64, true, false, true>, launch_pool<PathF64, true, true, true>}};
        const int f64 = p->precision == RRTB_PRECISION_F64;
        // motion: moving primitives under an open shutter, the kernels walk interpolating motion nodes
        const Launcher launch = ctx->lights ? (use_pool ? pool_lit[f64][ctx->motion] : lane_lit[f64][ctx->use_bvh != 0])
                                            : (use_pool ? pool[f64 ? 2 : ctx->n_mtriangles > 0][ctx->motion] : lane[f64][ctx->use_bvh != 0]);
        const int rc = launch(ctx, a, p->count_rays != 0, &blocks);
        if (rc) return rc;
        launches = 1;
    }
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    RRTB_CUDA(ctx, cudaGetLastError());
    ctx->pending = *p;
    ctx->pending_launches = launches;
    if (defer) return RRTB_OK; // the caller enqueues more work (other devices, the resolve) before finish_render
    return finish_render(ctx, stats);
}

// Waits for the render enqueued by launch_render and fills `stats` (device time by CUDA events on the context stream,
// counters of the counting build, camera paths of the shard).
int finish_render(rrtb_ctx *ctx, rrtb_stats *stats)
{
    const rrtb_render_params *p = &ctx->pending;
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    RRTB_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (stats) {
        stats->seconds_render = ms * 1e-3;
        stats->seconds_build = ctx->seconds_build;
        stats->seconds_resolve = 0.0;
        stats->kernel_launches = ctx->pending_launches;
        stats->rays = stats->box_tests = stats->sphere_tests = stats->msphere_tests = stats->triangle_tests = stats->hits = 0;
        if (p->count_rays) {
            unsigned long long c[8];
            RRTB_CUDA(ctx, cudaMemcpy(c, ctx->d_counters, sizeof(c), cudaMemcpyDeviceToHost));
            stats->rays = c[1];
            stats->box_tests = c[2];
            stats->sphere_tests = c[3];
            stats->msphere_tests = c[4];
            stats->triangle_tests = c[5];
            stats->hits = c[6];
        }
        // camera paths in this shard: its pixels (edge tiles are clipped) times its samples
        const ShardGeometry g = shard_geometry(p);
        unsigned long long px = 0;
        if (p->shard_mode == RRTB_SHARD_TILES && g.world > 1) {
            for (int t = g.rank; t < g.n_tiles; t += g.world) {
                int ty = t / g.tiles_x, tx = t - ty * g.tiles_x;
                int w = min(8, p->width - tx * 8), h = min(4, p->height - ty * 4);
                px += (unsigned long long)(w * h);
            }
        }
        else {
            px = (unsigned long long)p->width * p->height;
        }
        stats->paths = px * (unsigned long long)g.n_local_samples;
#ifdef RRTB_DEBUG_CHECKS
        unsigned int viol = 0;
        RRTB_CUDA(ctx, cudaMemcpyFromSymbol(&viol, g_rrtb_violations, sizeof(viol)));
        stats->reserved = (int32_t)viol; // cumulative count of violated invariants (debug build only)
#endif
    }
    return RRTB_OK;
}

// the AOV kernel: persistent, one wave, at most one warp per owned tile
template <class P, bool USE_BVH>
static int launch_aov_kernel(rrtb_ctx *ctx, const AovArgs &a, bool cnt)
{
    auto kernel = cnt ? k_render_aov<P, USE_BVH, true> : k_render_aov<P, USE_BVH, false>;
    int per_sm = 0;
    RRTB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, RENDER_TPB, 0));
    if (per_sm < 1) per_sm = 1;
    const int want = (a.n_local_tiles + RENDER_TPB / 32 - 1) / (RENDER_TPB / 32);
    const int blocks = min(ctx->sm_count * per_sm, max(want, 1));
    kernel<<<blocks, RENDER_TPB, 0, ctx->stream>>>(a);
    return RRTB_OK;
}

int launch_aov(rrtb_ctx *ctx, const rrtb_render_params *p, float *d_out, rrtb_stats *stats)
{
    const ShardGeometry g = shard_geometry(p); // p->shard_mode is RRTB_SHARD_TILES (rrtb_render_aov)
    AovArgs a;
    a.scene = device_scene(ctx);
    a.cam = device_camera(ctx->cam, p->width, p->height);
    a.W = p->width;
    a.H = p->height;
    a.spp = p->spp;
    a.key = make_uint2((uint32_t)p->seed, (uint32_t)(p->seed >> 32));
    a.rank = g.rank;
    a.world = g.world;
    a.tiles_x = g.tiles_x;
    a.n_local_tiles = g.n_local_tiles;
    a.out = d_out;
    a.queue = ctx->d_counters;
    RRTB_CUDA(ctx, cudaMemsetAsync(d_out, 0, 8 * sizeof(float) * (size_t)p->width * p->height, ctx->stream)); // pixels of other shards
    RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_counters, 0, 8 * sizeof(unsigned long long), ctx->stream));
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    typedef int (*Launcher)(rrtb_ctx *, const AovArgs &, bool);
    static const Launcher launch[2][2] = {{launch_aov_kernel<PathF32, false>, launch_aov_kernel<PathF32, true>},
                                          {launch_aov_kernel<PathF64, false>, launch_aov_kernel<PathF64, true>}};
    const int rc = launch[p->precision == RRTB_PRECISION_F64][ctx->use_bvh != 0](ctx, a, p->count_rays != 0);
    if (rc) return rc;
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    RRTB_CUDA(ctx, cudaGetLastError());
    ctx->pending = *p;
    ctx->pending_launches = 1;
    return finish_render(ctx, stats); // device time, counters and primary segments (stats.paths) as for a render
}

template <typename T>
int launch_resolve(rrtb_ctx *ctx, const uint64_t *d_accum, T *d_out, size_t n)
{
    k_resolve<T><<<grid_size(ctx, n), 256, 0, ctx->stream>>>((const unsigned long long *)d_accum, d_out, n);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}
template int launch_resolve<float>(rrtb_ctx *, const uint64_t *, float *, size_t);
template int launch_resolve<double>(rrtb_ctx *, const uint64_t *, double *, size_t);

int launch_resolve_tiles(rrtb_ctx *ctx, const uint64_t *d_accum, void *d_out, const rrtb_render_params *p, bool f64)
{
    const ShardGeometry g = shard_geometry(p);
    const int blocks = grid_size(ctx, 32 * (size_t)g.n_local_tiles); // one warp per owned tile
    if (f64)
        k_resolve_tiles<double><<<blocks, 256, 0, ctx->stream>>>((const unsigned long long *)d_accum, (double *)d_out, p->width, p->height,
                                                                 g.tiles_x, g.n_tiles, g.rank, g.world);
    else
        k_resolve_tiles<float><<<blocks, 256, 0, ctx->stream>>>((const unsigned long long *)d_accum, (float *)d_out, p->width, p->height,
                                                                g.tiles_x, g.n_tiles, g.rank, g.world);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}

int launch_accumulate_atomic(rrtb_ctx *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t n)
{
    k_accumulate_atomic<<<grid_size(ctx, n), 256, 0, ctx->stream>>>((unsigned long long *)d_dst, (const unsigned long long *)d_src, n);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}

int launch_accumulate(rrtb_ctx *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t n)
{
    k_accumulate<<<grid_size(ctx, n), 256, 0, ctx->stream>>>((unsigned long long *)d_dst, (const unsigned long long *)d_src, n);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}

template <typename real>
int launch_trace(rrtb_ctx *ctx, const real *d_rays7, int n, real t_min, int mode, int32_t *d_id, real *d_t, real *d_rec7)
{
    if (n <= 0) return RRTB_OK;
    k_trace<PathOf<real>><<<(n + 127) / 128, 128, 0, ctx->stream>>>(device_scene(ctx), d_rays7, n, t_min, mode, d_id, d_t, d_rec7);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}
template int launch_trace<float>(rrtb_ctx *, const float *, int, float, int, int32_t *, float *, float *);
template int launch_trace<double>(rrtb_ctx *, const double *, int, double, int, int32_t *, double *, double *);

template <typename real>
int launch_camera_rays(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *d_pix, int n, int sample, real *d_rays7)
{
    if (n <= 0) return RRTB_OK;
    uint2 key = make_uint2((uint32_t)p->seed, (uint32_t)(p->seed >> 32));
    k_camera_rays<PathOf<real>><<<(n + 127) / 128, 128, 0, ctx->stream>>>(device_camera(ctx->cam, p->width, p->height), p->width,
                                                                          p->height, key, d_pix, n, sample, d_rays7);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}
template int launch_camera_rays<float>(rrtb_ctx *, const rrtb_render_params *, const int32_t *, int, int, float *);
template int launch_camera_rays<double>(rrtb_ctx *, const rrtb_render_params *, const int32_t *, int, int, double *);

int launch_philox(rrtb_ctx *ctx, const uint32_t *d_ctr, int n, uint32_t k0, uint32_t k1, uint32_t *d_out)
{
    if (n <= 0) return RRTB_OK;
    k_philox<<<(n + 127) / 128, 128, 0, ctx->stream>>>(d_ctr, n, make_uint2(k0, k1), d_out);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}

template <typename real>
int launch_scatter(rrtb_ctx *ctx, const real *d_in16, const uint32_t *d_rnd4, int n, real *d_out8)
{
    if (n <= 0) return RRTB_OK;
    k_scatter_test<PathOf<real>><<<(n + 127) / 128, 128, 0, ctx->stream>>>(device_scene(ctx), d_in16, d_rnd4, n, d_out8);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}
template int launch_scatter<float>(rrtb_ctx *, const float *, const uint32_t *, int, float *);
template int launch_scatter<double>(rrtb_ctx *, const double *, const uint32_t *, int, double *);

} // namespace rrtb
