// rrtb_bvh.cu -- GPU-built LBVH for the rrt hot path (sm_100a).
//
// Replaces create_world<<<1,1>>> (rrt.cu:124-174) and the single-thread recursive median-split
// bvh_node constructor with its O(n^2) dev_sort (bvh.h:65-78,81-159).  Pipeline (all on the device,
// every stage a grid-wide kernel, no host round trips):
//
//   k_prepare      raw scene structs -> 48-byte leaf records, per-primitive AABB (sphere.h:60-64,
//                  moving_sphere.h:60-66 over the camera shutter, triangle.h:77-87), block partials of
//                  the centroid bounds
//   k_bounds       final reduction -> centroid lo, 1/extent, traversal box padding
//   k_morton       30-bit Morton code of the centroid, 64-bit key = code << 32 | object id
//   radix sort     4 stable LSD passes of 8 bits over the code (k_hist / k_scan / k_scatter)
//   k_karras       Karras 2012 internal nodes from the sorted keys (delta = clz64 of key xor)
//   k_refit        bottom-up boxes, second arrival at a node computes it (fminf/fmaxf: order independent)
//   k_collapse4    the 4-wide traversal tree: 128-byte nodes, padded child boxes as centre + half extent
//   k_flatten_leaves  leaf-ordered 48-byte primitive records
//
// Every floating-point step that feeds the Morton code uses explicit _rn intrinsics so the codes, the
// permutation and the topology are BIT-EXACT against oracle/rrt_oracle.c (tests/test_lbvh_parity.py).
#include "rrtb_internal.h"

#include <cuda_fp16.h>

#include <math.h>
#include <stdio.h>

namespace rrtb {

static constexpr int TPB = 256;
// layout of the small constant block that lives at the end of d_reduce
struct BuildConsts {
    float lo[3];
    float inv[3];
    float pad;
    float mag;
};

__device__ __forceinline__ float warp_min(float v)
{
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// (base, rate) of a coordinate that moves by `move` over dt starting from x at time0; a zero rate keeps x exactly
__device__ __forceinline__ void lin_of(float x_at_time0, float move, float dt, float time0, float &base, float &rate)
{
    rate = __fdiv_rn(move, dt);
    base = rate == 0.0f ? x_at_time0 : __fmaf_rn(-rate, time0, x_at_time0);
}

// One thread per object id.  partial[b*7 + 0..2] = centroid min, 3..5 = centroid max, 6 = max |coordinate|
__global__ void __launch_bounds__(TPB) k_prepare(const rrtb_sphere *__restrict__ sph, int ns,
                                                  const rrtb_msphere *__restrict__ msph, int nms,
                                                  const rrtb_triangle *__restrict__ tri, int nt,
                                                  const rrtb_mtriangle *__restrict__ mtri, int nmt, float cam_t0,
                                                  float cam_t1, float4 *__restrict__ prim, float4 *__restrict__ ext, int2 *__restrict__ info,
                                                  float *__restrict__ prim_box, float *__restrict__ prim_box01,
                                                  float *__restrict__ partial)
{
    const int n = ns + nms + nt + nmt;
    const int id = blockIdx.x * TPB + threadIdx.x;
    const float inf = __int_as_float(0x7f800000);
    float mn[3] = {inf, inf, inf}, mx[3] = {-inf, -inf, -inf};
    if (id < n) {
        float4 a, b = make_float4(0, 0, 0, 0), c = make_float4(0, 0, 0, 0);
        int mat;
        // boxes of the primitive at the two ENDS of the shutter (prim_box01, scenes with motion only): lo/hi at camera
        // time0 in e0, at time1 in e1; static primitives fill them from their one box below
        float e0[6], e1x[6];
        bool moving = false;
        if (id < ns) {
            rrtb_sphere s = sph[id];
            a = make_float4(s.center[0], s.center[1], s.center[2], s.radius);
            {
                // centre and radius once more as doubles, for the leaf test (rrtb_device.cuh sphere_test_d4): the record has
                // 32 spare bytes and the conversion (exact) then happens here instead of at every test
                const double d[4] = {(double)s.center[0], (double)s.center[1], (double)s.center[2], (double)s.radius};
                b = make_float4(__int_as_float(__double2loint(d[0])), __int_as_float(__double2hiint(d[0])),
                                __int_as_float(__double2loint(d[1])), __int_as_float(__double2hiint(d[1])));
                c = make_float4(__int_as_float(__double2loint(d[2])), __int_as_float(__double2hiint(d[2])),
                                __int_as_float(__double2loint(d[3])), __int_as_float(__double2hiint(d[3])));
            }
            mat = s.material;
            // sphere.h:60-64 with |radius|: the reference's center -+ radius is an INVERTED box for the negative radii the
            // book uses for hollow glass (its bvh then loses the sphere while the flat scan renders it); for radius >= 0
            // this is the reference's box bit for bit
            const float ar = fabsf(s.radius);
            for (int k = 0; k < 3; ++k) {
                mn[k] = __fsub_rn(s.center[k], ar);
                mx[k] = __fadd_rn(s.center[k], ar);
            }
        }
        else if (id < ns + nms) {
            rrtb_msphere m = msph[id - ns];
            float dt = __fsub_rn(m.time1, m.time0);
            float k0 = __fdiv_rn(__fsub_rn(cam_t0, m.time0), dt);
            float k1 = __fdiv_rn(__fsub_rn(cam_t1, m.time0), dt);
            float dc[3];
            const float ar = fabsf(m.radius);
            for (int k = 0; k < 3; ++k) {
                dc[k] = __fsub_rn(m.center1[k], m.center0[k]);
                float ca = __fadd_rn(m.center0[k], __fmul_rn(k0, dc[k]));
                float cb = __fadd_rn(m.center0[k], __fmul_rn(k1, dc[k]));
                mn[k] = fminf(__fsub_rn(ca, ar), __fsub_rn(cb, ar));
                mx[k] = fmaxf(__fadd_rn(ca, ar), __fadd_rn(cb, ar));
                e0[k] = __fsub_rn(ca, ar);
                e0[3 + k] = __fadd_rn(ca, ar);
                e1x[k] = __fsub_rn(cb, ar);
                e1x[3 + k] = __fadd_rn(cb, ar);
            }
            moving = true;
            a = make_float4(m.center0[0], m.center0[1], m.center0[2], m.radius);
            b = make_float4(dc[0], dc[1], dc[2], m.time0);
            c = make_float4(dt, 0.f, 0.f, 0.f);
            mat = m.material;
        }
        else if (id < ns + nms + nt) {
            rrtb_triangle t = tri[id - ns - nms];
            float e1[3], e2[3];
            for (int k = 0; k < 3; ++k) {
                e1[k] = __fsub_rn(t.v1[k], t.v0[k]);
                e2[k] = __fsub_rn(t.v2[k], t.v0[k]);
                mn[k] = fminf(fminf(t.v0[k], t.v1[k]), t.v2[k]);
                mx[k] = fmaxf(fmaxf(t.v0[k], t.v1[k]), t.v2[k]);
            }
            float nx, ny, nz;
            triangle_unit_normal(e1[0], e1[1], e1[2], e2[0], e2[1], e2[2], nx, ny, nz);
            a = make_float4(t.v0[0], t.v0[1], t.v0[2], nx);
            b = make_float4(e1[0], e1[1], e1[2], ny);
            c = make_float4(e2[0], e2[1], e2[2], nz);
            mat = t.material;
        }
        else { // SURVEY 8f4: triangle of a moving instance, include/rrtb.h "rrtb_mtriangle"
            rrtb_mtriangle t = mtri[id - ns - nms - nt];
            float dt = __fsub_rn(t.time1, t.time0);
            float base[3], rate[3], e1b[3], e1r[3], e2b[3], e2r[3];
            for (int k = 0; k < 3; ++k) {
                lin_of(t.v0[k], t.delta[k], dt, t.time0, base[k], rate[k]);
                lin_of(__fsub_rn(t.v1[k], t.v0[k]), t.extra1[k], dt, t.time0, e1b[k], e1r[k]);
                lin_of(__fsub_rn(t.v2[k], t.v0[k]), t.extra2[k], dt, t.time0, e2b[k], e2r[k]);
                // union of the poses at the two ends of the shutter, T = camera time0 / time1: {v0(T), v0(T)+e1(T), v0(T)+e2(T)};
                // motion is linear in time, so they bound every pose in between
                float pa = __fmaf_rn(rate[k], cam_t0, base[k]), pb = __fmaf_rn(rate[k], cam_t1, base[k]);
                float a1 = lin_at(e1r[k], cam_t0, e1b[k]), a2 = lin_at(e2r[k], cam_t0, e2b[k]);
                float b1 = lin_at(e1r[k], cam_t1, e1b[k]), b2 = lin_at(e2r[k], cam_t1, e2b[k]);
                e0[k] = fminf(fminf(pa, __fadd_rn(pa, a1)), __fadd_rn(pa, a2));
                e0[3 + k] = fmaxf(fmaxf(pa, __fadd_rn(pa, a1)), __fadd_rn(pa, a2));
                e1x[k] = fminf(fminf(pb, __fadd_rn(pb, b1)), __fadd_rn(pb, b2));
                e1x[3 + k] = fmaxf(fmaxf(pb, __fadd_rn(pb, b1)), __fadd_rn(pb, b2));
                mn[k] = fminf(e0[k], e1x[k]);
                mx[k] = fmaxf(e0[3 + k], e1x[3 + k]);
            }
            moving = true;
            a = make_float4(base[0], base[1], base[2], rate[0]);
            b = make_float4(e1b[0], e1b[1], e1b[2], rate[1]);
            c = make_float4(e2b[0], e2b[1], e2b[2], rate[2]);
            ext[2 * id + 0] = make_float4(e1r[0], e1r[1], e1r[2], 0.f);
            ext[2 * id + 1] = make_float4(e2r[0], e2r[1], e2r[2], 0.f);
            mat = t.material;
        }
        prim[3 * id + 0] = a;
        prim[3 * id + 1] = b;
        prim[3 * id + 2] = c;
        info[id] = make_int2(id, mat);
        for (int k = 0; k < 3; ++k) {
            prim_box[6 * id + k] = mn[k];
            prim_box[6 * id + 3 + k] = mx[k];
        }
        if (prim_box01)
            for (int k = 0; k < 3; ++k) {
                prim_box01[12 * id + k] = moving ? e0[k] : mn[k];
                prim_box01[12 * id + 3 + k] = moving ? e0[3 + k] : mx[k];
                prim_box01[12 * id + 6 + k] = moving ? e1x[k] : mn[k];
                prim_box01[12 * id + 9 + k] = moving ? e1x[3 + k] : mx[k];
            }
    }
    // block reduction of centroid bounds and coordinate magnitude
    float v[7];
    if (id < n) {
        float mag = 0.f;
        for (int k = 0; k < 3; ++k) {
            float cen = __fmul_rn(0.5f, __fadd_rn(mn[k], mx[k]));
            v[k] = cen;
            v[3 + k] = cen;
            mag = fmaxf(mag, fmaxf(fabsf(mn[k]), fabsf(mx[k])));
        }
        v[6] = mag;
    }
    else {
        for (int k = 0; k < 3; ++k) {
            v[k] = inf;
            v[3 + k] = -inf;
        }
        v[6] = 0.f;
    }
    __shared__ float sh[7][TPB / 32];
    for (int k = 0; k < 7; ++k) {
        float r = k < 3 ? warp_min(v[k]) : warp_max(v[k]);
        if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = r;
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        int k = threadIdx.x;
        float r = sh[k][0];
        for (int w = 1; w < TPB / 32; ++w) r = k < 3 ? fminf(r, sh[k][w]) : fmaxf(r, sh[k][w]);
        partial[blockIdx.x * 7 + k] = r;
    }
}

// single block: reduce the per-block partials, derive the Morton normalisation and the box padding
__global__ void __launch_bounds__(TPB) k_bounds(const float *__restrict__ partial, int nblocks, float cam_mag,
                                                 BuildConsts *__restrict__ out)
{
    const float inf = __int_as_float(0x7f800000);
    float v[7];
    for (int k = 0; k < 7; ++k) v[k] = k < 3 ? inf : (k < 6 ? -inf : 0.f);
    for (int b = threadIdx.x; b < nblocks; b += TPB)
        for (int k = 0; k < 7; ++k) {
            float x = partial[b * 7 + k];
            v[k] = k < 3 ? fminf(v[k], x) : fmaxf(v[k], x);
        }
    __shared__ float sh[7][TPB / 32];
    for (int k = 0; k < 7; ++k) {
        float r = k < 3 ? warp_min(v[k]) : warp_max(v[k]);
        if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = r;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float r[7];
        for (int k = 0; k < 7; ++k) {
            r[k] = sh[k][0];
            for (int w = 1; w < TPB / 32; ++w) r[k] = k < 3 ? fminf(r[k], sh[k][w]) : fmaxf(r[k], sh[k][w]);
        }
        for (int k = 0; k < 3; ++k) {
            float ext = __fsub_rn(r[3 + k], r[k]);
            out->lo[k] = r[k];
            out->inv[k] = ext > 0.f ? __fdiv_rn(1.0f, ext) : 0.f;
        }
        float mag = fmaxf(r[6], cam_mag);
        out->mag = mag;
        out->pad = __fmul_rn(mag, 9.5367431640625e-07f); // 2^-20 * largest coordinate magnitude
    }
}

__device__ __forceinline__ uint32_t expand_bits10(uint32_t v)
{
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__global__ void __launch_bounds__(TPB) k_morton(const float *__restrict__ prim_box, int n,
                                                 const BuildConsts *__restrict__ bc, uint32_t *__restrict__ morton,
                                                 uint64_t *__restrict__ keys)
{
    int id = blockIdx.x * TPB + threadIdx.x;
    if (id >= n) return;
    uint32_t q[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float cen = __fmul_rn(0.5f, __fadd_rn(prim_box[6 * id + k], prim_box[6 * id + 3 + k]));
        float x = __fmul_rn(__fsub_rn(cen, bc->lo[k]), bc->inv[k]);
        int v = (int)__fmul_rn(x, 1024.0f); // truncation toward zero, as the C cast
        v = v < 0 ? 0 : (v > 1023 ? 1023 : v);
        q[k] = (uint32_t)v;
    }
    uint32_t code = (expand_bits10(q[0]) << 2) | (expand_bits10(q[1]) << 1) | expand_bits10(q[2]);
    morton[id] = code;
    keys[id] = ((uint64_t)code << 32) | (uint32_t)id;
}

// ---- stable LSD radix sort, 8 bits per pass ---------------------------------------------------------
// Each WARP owns a contiguous segment of SEG keys, so the global order of (segment, position) is the
// input order and stability falls out of processing a segment front to back.
static constexpr int SEG = 1024;           // keys per warp
static constexpr int SORT_WARPS = TPB / 32; // warps per block

__global__ void __launch_bounds__(TPB) k_hist(const uint64_t *__restrict__ keys, int n, int shift, int n_seg,
                                               unsigned int *__restrict__ hist)
{
    __shared__ unsigned int sh[SORT_WARPS][256];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int seg = blockIdx.x * SORT_WARPS + w;
    for (int d = lane; d < 256; d += 32) sh[w][d] = 0;
    __syncwarp();
    if (seg < n_seg) {
        const int beg = seg * SEG, end = min(beg + SEG, n);
        for (int i = beg + lane; i < end; i += 32) atomicAdd(&sh[w][(unsigned)(keys[i] >> shift) & 255u], 1u);
        __syncwarp();
        for (int d = lane; d < 256; d += 32) hist[d * n_seg + seg] = sh[w][d];
    }
}

// Exclusive scan of hist[256 * n_seg] (digit-major) in three grid-wide steps: per-chunk sums, a scan of the chunk
// sums (one block; <= a few hundred values for a million primitives), per-chunk exclusive scans offset by them.
// (One block walking the whole array took 0.23 ms per pass at 1.1 M primitives -- over half of the build.)
static constexpr int SCAN_CHUNK = 4096; // entries per block: 256 threads x 16

__device__ __forceinline__ unsigned int block_exclusive_scan_256(unsigned int v, unsigned int *warp_sums, unsigned int &total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned int incl = v;
    for (int o = 1; o < 32; o <<= 1) {
        unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[w] = incl;
    __syncthreads();
    if (w == 0) {
        unsigned int s = lane < TPB / 32 ? warp_sums[lane] : 0u;
        unsigned int si = s;
        for (int o = 1; o < 32; o <<= 1) {
            unsigned int t = __shfl_up_sync(0xffffffffu, si, o);
            if (lane >= o) si += t;
        }
        if (lane < TPB / 32) warp_sums[lane] = si - s; // exclusive prefix of the warp sums
        if (lane == 31) warp_sums[TPB / 32] = si;       // block total
    }
    __syncthreads();
    total = warp_sums[TPB / 32];
    return warp_sums[w] + incl - v;
}

__global__ void __launch_bounds__(TPB) k_scan_sums(const unsigned int *__restrict__ hist, int total, unsigned int *__restrict__ sums)
{
    __shared__ unsigned int warp_sums[TPB / 32 + 1];
    const int base = blockIdx.x * SCAN_CHUNK + threadIdx.x * 16;
    unsigned int v = 0;
    for (int k = 0; k < 16; ++k)
        if (base + k < total) v += hist[base + k];
    unsigned int tot;
    block_exclusive_scan_256(v, warp_sums, tot);
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(TPB) k_scan_apply(unsigned int *__restrict__ hist, int total, const unsigned int *__restrict__ sums)
{
    __shared__ unsigned int warp_sums[TPB / 32 + 1];
    const int base = blockIdx.x * SCAN_CHUNK + threadIdx.x * 16;
    unsigned int x[16], v = 0;
    for (int k = 0; k < 16; ++k) {
        x[k] = base + k < total ? hist[base + k] : 0u;
        v += x[k];
    }
    unsigned int tot;
    unsigned int run = sums[blockIdx.x] + block_exclusive_scan_256(v, warp_sums, tot);
    for (int k = 0; k < 16; ++k) {
        if (base + k < total) hist[base + k] = run;
        run += x[k];
    }
}

// exclusive scan of a short array in place, single block (the chunk sums)
__global__ void __launch_bounds__(1024) k_scan(unsigned int *__restrict__ hist, int total)
{
    __shared__ unsigned int warp_sums[32];
    __shared__ unsigned int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int base = 0; base < total; base += 1024) {
        int i = base + threadIdx.x;
        unsigned int v = i < total ? hist[i] : 0u;
        unsigned int incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sums[w] = incl;
        __syncthreads();
        if (w == 0) {
            unsigned int s = warp_sums[lane];
            unsigned int si = s;
            for (int o = 1; o < 32; o <<= 1) {
                unsigned int t = __shfl_up_sync(0xffffffffu, si, o);
                if (lane >= o) si += t;
            }
            warp_sums[lane] = si - s; // exclusive prefix of warp sums
        }
        __syncthreads();
        unsigned int excl = carry + warp_sums[w] + incl - v;
        if (i < total) hist[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(TPB) k_scatter(const uint64_t *__restrict__ in, uint64_t *__restrict__ out, int n,
                                                  int shift, int n_seg, const unsigned int *__restrict__ hist)
{
    __shared__ unsigned int off[SORT_WARPS][256];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int seg = blockIdx.x * SORT_WARPS + w;
    if (seg >= n_seg) return;
    for (int d = lane; d < 256; d += 32) off[w][d] = hist[d * n_seg + seg];
    __syncwarp();
    const int beg = seg * SEG, end = min(beg + SEG, n);
    for (int base = beg; base < end; base += 32) {
        int i = base + lane;
        bool valid = i < end;
        unsigned int active = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            uint64_t key = in[i];
            unsigned int d = (unsigned)(key >> shift) & 255u;
            unsigned int peers = __match_any_sync(active, d);
            unsigned int rank = __popc(peers & ((1u << lane) - 1u));
            unsigned int pos = off[w][d] + rank;
            out[pos] = key;
            __syncwarp(active);
            if (rank == 0) off[w][d] += __popc(peers);
        }
        __syncwarp();
    }
}

// Scenes of at most SMALL_SORT keys (the reference's four scenes have 4 .. 488 primitives) are sorted by ONE block in
// shared memory: a bitonic network over the whole 64-bit key.  Keys are unique (the id is in the low word), so the
// result is the order the stable radix passes produce; 20 launches of ~5 us each become one.
static constexpr int SMALL_SORT = 2048;

__global__ void __launch_bounds__(1024) k_sort_small(uint64_t *__restrict__ keys, int n)
{
    __shared__ uint64_t sk[SMALL_SORT];
    int m = 2;
    while (m < n) m <<= 1; // padded length
    for (int i = threadIdx.x; i < m; i += 1024) sk[i] = i < n ? keys[i] : ~0ull;
    __syncthreads();
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < (m >> 1); t += 1024) {
                const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j; // the t-th pair at distance j
                const bool up = (lo & k) == 0;
                const uint64_t a = sk[lo], b = sk[hi];
                if ((a > b) == up) {
                    sk[lo] = b;
                    sk[hi] = a;
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < n; i += 1024) keys[i] = sk[i];
}

// ---- Karras 2012 ------------------------------------------------------------------------------------
__device__ __forceinline__ int delta_fn(const uint64_t *__restrict__ keys, int n, uint64_t ki, int j)
{
    if (j < 0 || j >= n) return -1;
    return __clzll((long long)(ki ^ keys[j]));
}

__global__ void __launch_bounds__(TPB) k_karras(const uint64_t *__restrict__ keys, int n, int *__restrict__ left,
                                                 int *__restrict__ right, int *__restrict__ parent, int2 *__restrict__ range)
{
    const int i = blockIdx.x * TPB + threadIdx.x;
    const int ni = n - 1;
    if (i >= ni) return;
    const uint64_t ki = keys[i];
    int d = (delta_fn(keys, n, ki, i + 1) - delta_fn(keys, n, ki, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta_fn(keys, n, ki, i - d);
    int lmax = 2;
    while (delta_fn(keys, n, ki, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (delta_fn(keys, n, ki, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta_fn(keys, n, ki, j);
    int s = 0;
    int t = l;
    do {
        t = (t + 1) >> 1;
        if (delta_fn(keys, n, ki, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + (d < 0 ? -1 : 0);
    int mn = min(i, j), mx = max(i, j);
    int L = (mn == gamma) ? ~gamma : gamma;
    int R = (mx == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    left[i] = L;
    right[i] = R;
    range[i] = make_int2(mn, mx); // the sorted positions this node covers (its internal nodes are mn .. mx - 1)
    parent[L >= 0 ? L : (ni + ~L)] = i;
    parent[R >= 0 ? R : (ni + ~R)] = i;
    if (i == 0) parent[0] = -1;
}

// ---- SAH rebuild of the lower tree (traversal structure only; the canonical LBVH above stays as it is) ---------------
// Every maximal subtree of the Karras tree with at most SAH_MAX leaves is rebuilt top-down with the binned surface-area
// heuristic by one thread block: the leaves of a Karras node are a contiguous run of sorted positions and its internal
// nodes are the indices strictly inside that run, so the new subtree is written into the SAME node slots (the subtree
// root keeps its index, hence its parent's link).  A scene of up to SAH_MAX primitives is rebuilt whole.  Measured on recorded ray
// populations (tools/treelab): -8.5 % visits of the 4-wide tree on final.txt and on the 1.1 M-primitive scene.
// Level-synchronous inside the block: a warp takes a task (node, run of leaves), bins the leaves' centroids along the
// three axes (shared-memory atomics), evaluates the 31 candidate planes of each axis with one lane each (prefix and
// suffix unions of the bins by warp scans), partitions the run into the
// other index buffer and emits the two children; runs of one leaf become leaf children at once.
static constexpr int SAH_MAX = 512;
static constexpr int SAH_BINS = 32; // one bin per lane: prefix / suffix unions by warp scans (tools/treelab: 8 bins -4.8 %, 16 -6.8 %, 32 -12 % visits on final.txt)
static constexpr int SAH_BIG = 128; // runs longer than this are split by the whole block (blocks of at least SAH_MAX threads only)

struct SahState {
    int n_roots; // subtrees to rebuild
    int ticket;  // next one to hand out
};

__global__ void __launch_bounds__(TPB) k_sah_select(int n, const int *__restrict__ left, const int *__restrict__ right,
                                                     const int *__restrict__ parent, const int2 *__restrict__ range,
                                                     int *__restrict__ left2, int *__restrict__ right2, int *__restrict__ parent2,
                                                     int *__restrict__ roots, SahState *st)
{
    const int i = blockIdx.x * TPB + threadIdx.x;
    const int ni = n - 1;
    if (i < 2 * n - 1) parent2[i] = parent[i];
    if (i >= ni) return;
    left2[i] = left[i];
    right2[i] = right[i];
    const int size = range[i].y - range[i].x + 1;
    const int p = parent[i];
    const int psize = p >= 0 ? range[p].y - range[p].x + 1 : 0x7fffffff;
    if (size >= 3 && size <= SAH_MAX && psize > SAH_MAX) roots[atomicAdd(&st->n_roots, 1)] = i;
}

// The arithmetic of the SAH rebuild and of the collapse, written so that each product, sum and quotient rounds once:
// ptxas would otherwise contract products and sums into FMAs where it chooses, and the tree would then depend on the
// compiler.  oracle/rrt_oracle_wide.c restates these definitions as plain C built with -ffp-contract=off.
//   area_rn      x*y + y*z + z*x, half the surface area of a box of extents x, y, z
//   sah_cost_rn  a0*n0 + a1*n1, the SAH cost of a split into boxes of areas a0, a1 holding n0, n1 primitives
//   sah_bin      the bin of twice a centroid, c2 = lo + hi, among SAH_BINS over [cmin, cmin + SAH_BINS / scale]
__device__ __forceinline__ float area_rn(float x, float y, float z)
{
    return __fadd_rn(__fadd_rn(__fmul_rn(x, y), __fmul_rn(y, z)), __fmul_rn(z, x));
}
__device__ __forceinline__ float sah_cost_rn(float a0, int n0, float a1, int n1)
{
    return __fadd_rn(__fmul_rn(a0, (float)n0), __fmul_rn(a1, (float)n1));
}
__device__ __forceinline__ float centroid2(const float *box, int k) { return __fadd_rn(box[k], box[3 + k]); }
__device__ __forceinline__ float sah_scale(float cmin, float cmax) { return cmax > cmin ? __fdiv_rn((float)SAH_BINS, __fsub_rn(cmax, cmin)) : 0.f; }
__device__ __forceinline__ int sah_bin(float c2, float cmin, float scale) { return min(SAH_BINS - 1, (int)__fmul_rn(__fsub_rn(c2, cmin), scale)); }

// order-preserving float <-> int (for atomicMin / atomicMax on shared memory)
__device__ __forceinline__ int f2o(float f)
{
    const int b = __float_as_int(f);
    return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float o2f(int o) { return __int_as_float(o >= 0 ? o : o ^ 0x7fffffff); }

// Best split of one task from its bins (lane = bin): the plane after bin `lane` splits the run into bins 0 .. lane and
// lane + 1 .. 31; their unions by an inclusive prefix scan and an exclusive suffix scan over the lanes.  Returns, in every
// lane, the cheapest (cost, axis * 32 + bin); cost = +inf when no plane has primitives on both sides.  Lane 31 also gets
// the box of the whole run (the last inclusive prefix) in `whole`.
__device__ __forceinline__ void sah_choose(const int (*bn3)[SAH_BINS][7], int lane, float &cost, int &best, float *whole)
{
    const float inf = __int_as_float(0x7f800000);
    cost = inf;
    best = 0;
    for (int k = 0; k < 3; ++k) {
        const int *bn = bn3[k][lane];
        int pc = bn[0];
        float plo[3], phi[3];
        for (int c = 0; c < 3; ++c) {
            plo[c] = o2f(bn[1 + c]);
            phi[c] = o2f(bn[4 + c]);
        }
        int sc = pc;
        float slo[3] = {plo[0], plo[1], plo[2]}, shi[3] = {phi[0], phi[1], phi[2]};
        for (int o = 1; o < 32; o <<= 1) {
            const int c_up = __shfl_up_sync(0xffffffffu, pc, o), c_dn = __shfl_down_sync(0xffffffffu, sc, o);
            if (lane >= o) pc += c_up;
            if (lane + o < 32) sc += c_dn;
            for (int c = 0; c < 3; ++c) {
                const float lu = __shfl_up_sync(0xffffffffu, plo[c], o), hu = __shfl_up_sync(0xffffffffu, phi[c], o);
                const float ld = __shfl_down_sync(0xffffffffu, slo[c], o), hd = __shfl_down_sync(0xffffffffu, shi[c], o);
                if (lane >= o) {
                    plo[c] = fminf(plo[c], lu);
                    phi[c] = fmaxf(phi[c], hu);
                }
                if (lane + o < 32) {
                    slo[c] = fminf(slo[c], ld);
                    shi[c] = fmaxf(shi[c], hd);
                }
            }
        }
        if (k == 0)
            for (int c = 0; c < 3; ++c) {
                whole[c] = plo[c];
                whole[3 + c] = phi[c];
            }
        // the right side of the plane after bin `lane` is the inclusive suffix of lane + 1
        const int rc = __shfl_down_sync(0xffffffffu, sc, 1);
        float rlo[3], rhi[3];
        for (int c = 0; c < 3; ++c) {
            rlo[c] = __shfl_down_sync(0xffffffffu, slo[c], 1);
            rhi[c] = __shfl_down_sync(0xffffffffu, shi[c], 1);
        }
        if (lane < 31 && pc > 0 && rc > 0) {
            const float a0 = area_rn(__fsub_rn(phi[0], plo[0]), __fsub_rn(phi[1], plo[1]), __fsub_rn(phi[2], plo[2]));
            const float a1 = area_rn(__fsub_rn(rhi[0], rlo[0]), __fsub_rn(rhi[1], rlo[1]), __fsub_rn(rhi[2], rlo[2]));
            const float ck = sah_cost_rn(a0, pc, a1, rc);
            if (ck < cost) {
                cost = ck;
                best = k * 32 + lane;
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float oc = __shfl_xor_sync(0xffffffffu, cost, o);
        const int ob = __shfl_xor_sync(0xffffffffu, best, o);
        if (oc < cost || (oc == cost && ob < best)) {
            cost = oc;
            best = ob;
        }
    }
}

__device__ __forceinline__ void sah_bins_clear(int (*bn3)[SAH_BINS][7], int lane)
{
    const float inf = __int_as_float(0x7f800000);
    for (int k = 0; k < 3; ++k) { // lane = bin
        int *bn = bn3[k][lane];
        bn[0] = 0;
        for (int c = 0; c < 3; ++c) {
            bn[1 + c] = f2o(inf);
            bn[4 + c] = f2o(-inf);
        }
    }
}

__device__ __forceinline__ void sah_bins_add(int (*bn3)[SAH_BINS][7], const float *box, const float *cmin, const float *scale)
{
    for (int k = 0; k < 3; ++k) {
        int *bn = bn3[k][sah_bin(centroid2(box, k), cmin[k], scale[k])];
        atomicAdd(&bn[0], 1);
        for (int c3 = 0; c3 < 3; ++c3) {
            atomicMin(&bn[1 + c3], f2o(box[c3]));
            atomicMax(&bn[4 + c3], f2o(box[3 + c3]));
        }
    }
}

// One block rebuilds one subtree at a time, level by level.  Per level: tasks of more than SAH_BIG primitives (the top of
// the subtree: few tasks, long runs) are taken one after the other by the WHOLE block, one primitive per thread; the
// others by one warp each.  Two shapes: NT = 1024 for scenes of a few subtrees (the reference's scenes are ONE subtree: the
// build is a latency chain and every level wants all the warps it can get), NT = 256 with four blocks per SM and no
// block-wide path for large scenes, where there are thousands of subtrees to overlap (1.1 M primitives: 4.0 vs 5.2 ms).
template <int NT>
__global__ void __launch_bounds__(NT) k_sah_rebuild(const uint64_t *__restrict__ keys, int n, const int2 *__restrict__ range,
                                                          const float *__restrict__ prim_box, const int *__restrict__ roots,
                                                          const int *__restrict__ parent, SahState *st, int *__restrict__ left2,
                                                          int *__restrict__ right2, int *__restrict__ parent2, float *__restrict__ node_box2)
{
    constexpr int SAH_TPB = NT, SAH_WARPS = NT / 32;
    constexpr bool BLOCK_PATH = NT >= SAH_MAX; // one thread per primitive of a run
    extern __shared__ int sah_dyn[];
    int (*bins)[3][SAH_BINS][7] = reinterpret_cast<int (*)[3][SAH_BINS][7]>(sah_dyn); // [SAH_WARPS]: count, min xyz, max xyz (ordered ints)
    __shared__ float sbox[SAH_MAX][6];
    __shared__ unsigned short sidx[2][SAH_MAX];
    __shared__ int q_node[2][SAH_MAX / 2 + 1];
    __shared__ unsigned short q_b[2][SAH_MAX / 2 + 1], q_e[2][SAH_MAX / 2 + 1];
    __shared__ int q_n[2];
    __shared__ int s_alloc, s_root, s_budget;
    __shared__ int s_cmin[3], s_cmax[3], s_best, s_median, s_cl[SAH_WARPS], s_cr[SAH_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int ni = n - 1;
    const float inf = __int_as_float(0x7f800000);

    while (true) {
        __syncthreads();
        if (tid == 0) s_root = atomicAdd(&st->ticket, 1);
        __syncthreads();
        if (s_root >= st->n_roots) return;
        const int root = roots[s_root];
        const int a = range[root].x, m = range[root].y - range[root].x + 1;
        for (int l = tid; l < m; l += SAH_TPB) {
            const int id = (int)(uint32_t)keys[a + l];
            for (int c = 0; c < 6; ++c) sbox[l][c] = prim_box[6 * id + c];
            sidx[0][l] = (unsigned short)l;
        }
        if (tid == 0) {
            // The traversal stack (RRTB_STACK = 3 x 64 entries) relies on a tree of at most 63 levels, which the Karras tree
            // guarantees (30-bit codes + 32-bit index tie-break).  The rebuilt subtree gets the levels its root leaves free;
            // a run that could not be finished inside them by halving is split in the middle from there on.
            int d = 0;
            for (int p = parent[root]; p >= 0; p = parent[p]) ++d;
            s_budget = 63 - d;
            // A Karras node sits at one END of the run [a, a + m - 1] it covers and the internal nodes below it are the
            // indices strictly inside the run (the other end belongs to a node outside the subtree): m - 2 slots for the
            // m - 2 internal nodes below the root.
            s_alloc = a + 1;
            q_node[0][0] = root;
            q_b[0][0] = 0;
            q_e[0][0] = (unsigned short)m;
            q_n[0] = 1;
            q_n[1] = 0;
        }
        __syncthreads();
        int cur = 0, level = 0;
        // the two children of `node` over the partitioned run [b, b + nl) [b + nl, e) of sidx[cur ^ 1]: a run of one leaf is a
        // leaf child, a longer run a new node and a task of the next level (one thread)
        auto emit = [&](int node, int b, int nl, int e) {
            int child[2];
            const int cb[2] = {b, b + nl}, ce[2] = {b + nl, e};
            for (int sd = 0; sd < 2; ++sd) {
                if (ce[sd] - cb[sd] == 1) {
                    const int k = a + sidx[cur ^ 1][cb[sd]];
                    child[sd] = ~k;
                    parent2[ni + k] = node;
                }
                else {
                    const int v = atomicAdd(&s_alloc, 1);
                    child[sd] = v;
                    parent2[v] = node;
                    const int q = atomicAdd(&q_n[cur ^ 1], 1);
                    q_node[cur ^ 1][q] = v;
                    q_b[cur ^ 1][q] = (unsigned short)cb[sd];
                    q_e[cur ^ 1][q] = (unsigned short)ce[sd];
                }
            }
            left2[node] = child[0];
            right2[node] = child[1];
        };
        while (q_n[cur] > 0) {
            const int n_tasks = q_n[cur];
            // ---- long runs: the whole block, one primitive per thread (SAH_MAX <= SAH_TPB)
            for (int t = 0; BLOCK_PATH && t < n_tasks; ++t) {
                const int node = q_node[cur][t], b = q_b[cur][t], e = q_e[cur][t], cnt = e - b;
                if (cnt <= SAH_BIG) continue; // block-uniform
                if (tid < 3) {
                    s_cmin[tid] = f2o(inf);
                    s_cmax[tid] = f2o(-inf);
                }
                if (warp == 0) sah_bins_clear(bins[0], lane);
                __syncthreads();
                const bool valid = tid < cnt;
                const int l = valid ? sidx[cur][b + tid] : 0;
                float box[6];
                for (int c = 0; c < 6; ++c) box[c] = sbox[l][c];
                if (warp * 32 < cnt) { // centroid bounds (twice the centroid: lo + hi)
                    for (int k = 0; k < 3; ++k) {
                        const float c = centroid2(box, k);
                        const float mn = warp_min(valid ? c : inf), mx = warp_max(valid ? c : -inf);
                        if (lane == 0) {
                            atomicMin(&s_cmin[k], f2o(mn));
                            atomicMax(&s_cmax[k], f2o(mx));
                        }
                    }
                }
                __syncthreads();
                float cmin[3], scale[3];
                for (int k = 0; k < 3; ++k) {
                    const float cmax = o2f(s_cmax[k]);
                    cmin[k] = o2f(s_cmin[k]);
                    scale[k] = sah_scale(cmin[k], cmax);
                }
                if (valid) sah_bins_add(bins[0], box, cmin, scale);
                __syncthreads();
                if (warp == 0) {
                    float cost, whole[6];
                    int best;
                    sah_choose(bins[0], lane, cost, best, whole);
                    if (lane == 31)
                        for (int c = 0; c < 6; ++c) node_box2[6 * node + c] = whole[c];
                    if (lane == 0) {
                        s_best = best;
                        s_median = !(cost < inf) || level + (32 - __clz(cnt - 1)) >= s_budget;
                    }
                }
                __syncthreads();
                const int ax = s_best >> 5, sp = s_best & 31;
                bool go_left = false;
                if (valid) {
                    if (s_median) go_left = tid < cnt / 2;
                    else go_left = sah_bin(centroid2(box, ax), cmin[ax], scale[ax]) <= sp;
                }
                const unsigned ml = __ballot_sync(0xffffffffu, go_left), mr = __ballot_sync(0xffffffffu, valid && !go_left);
                if (lane == 0) {
                    s_cl[warp] = __popc(ml);
                    s_cr[warp] = __popc(mr);
                }
                __syncthreads();
                int offl = 0, offr = 0, nl = 0;
                for (int w = 0; w < SAH_WARPS; ++w) {
                    if (w < warp) {
                        offl += s_cl[w];
                        offr += s_cr[w];
                    }
                    nl += s_cl[w];
                }
                if (go_left) sidx[cur ^ 1][b + offl + __popc(ml & lt)] = (unsigned short)l;
                else if (valid) sidx[cur ^ 1][e - 1 - (offr + __popc(mr & lt))] = (unsigned short)l;
                __syncthreads();
                if (tid == 0) emit(node, b, nl, e);
            }
            // ---- the other runs: one warp each
            for (int t = warp; t < n_tasks; t += SAH_WARPS) {
                const int node = q_node[cur][t], b = q_b[cur][t], e = q_e[cur][t], cnt = e - b;
                if (BLOCK_PATH && cnt > SAH_BIG) continue;
                int nl = 0;
                if (cnt <= 4) {
                    // Two to four boxes: EVERY way to split them into two sets (2^(cnt-1) - 1 of them, element 0 on the left), one
                    // candidate per lane -- exact where the bins are coarsest, and most tasks of a subtree are this small.
                    float lo4[4][3], hi4[4][3];
                    for (int i = 0; i < 4; ++i) {
                        const int l = sidx[cur][b + min(i, cnt - 1)];
                        for (int c = 0; c < 3; ++c) {
                            lo4[i][c] = sbox[l][c];
                            hi4[i][c] = sbox[l][3 + c];
                        }
                    }
                    if (lane < 3) { // the node's own box: lanes 0..2 = axes
                        float lo = lo4[0][lane], hi = hi4[0][lane];
                        for (int i = 1; i < 4; ++i)
                            if (i < cnt) {
                                lo = fminf(lo, lo4[i][lane]);
                                hi = fmaxf(hi, hi4[i][lane]);
                            }
                        node_box2[6 * node + lane] = lo;
                        node_box2[6 * node + 3 + lane] = hi;
                    }
                    const unsigned mask = 1u | ((unsigned)lane << 1);
                    float cost = inf;
                    if (lane < (1 << (cnt - 1)) - 1) {
                        float alo[3] = {inf, inf, inf}, ahi[3] = {-inf, -inf, -inf}, blo[3] = {inf, inf, inf}, bhi[3] = {-inf, -inf, -inf};
                        for (int i = 0; i < 4; ++i) {
                            if (i >= cnt) break;
                            const bool left = (mask >> i) & 1u;
                            for (int c = 0; c < 3; ++c) {
                                if (left) {
                                    alo[c] = fminf(alo[c], lo4[i][c]);
                                    ahi[c] = fmaxf(ahi[c], hi4[i][c]);
                                }
                                else {
                                    blo[c] = fminf(blo[c], lo4[i][c]);
                                    bhi[c] = fmaxf(bhi[c], hi4[i][c]);
                                }
                            }
                        }
                        const int na = __popc(mask & ((1u << cnt) - 1u));
                        const float a0 = area_rn(__fsub_rn(ahi[0], alo[0]), __fsub_rn(ahi[1], alo[1]), __fsub_rn(ahi[2], alo[2]));
                        const float a1 = area_rn(__fsub_rn(bhi[0], blo[0]), __fsub_rn(bhi[1], blo[1]), __fsub_rn(bhi[2], blo[2]));
                        cost = sah_cost_rn(a0, na, a1, cnt - na);
                    }
                    int best = lane;
                    for (int o = 4; o > 0; o >>= 1) {
                        const float oc = __shfl_xor_sync(0xffffffffu, cost, o);
                        const int ob = __shfl_xor_sync(0xffffffffu, best, o);
                        if (oc < cost || (oc == cost && ob < best)) {
                            cost = oc;
                            best = ob;
                        }
                    }
                    best = __shfl_sync(0xffffffffu, best, 0);
                    cost = __shfl_sync(0xffffffffu, cost, 0);
                    unsigned bm = 1u | ((unsigned)best << 1);
                    // no finite candidate, or an uneven split could outgrow the depth budget: halve
                    if (!(cost < inf) || level + cnt - 1 >= s_budget) bm = (1u << (cnt / 2)) - 1u;
                    nl = __popc(bm);
                    if (lane < cnt) {
                        const bool left = (bm >> lane) & 1u;
                        const int pos = left ? __popc(bm & lt) : nl + __popc(~bm & lt);
                        sidx[cur ^ 1][b + pos] = sidx[cur][b + lane];
                    }
                    __syncwarp();
                }
                else {
                    // centroid bounds (twice the centroid: lo + hi)
                    float cmin[3] = {inf, inf, inf}, cmax[3] = {-inf, -inf, -inf};
                    for (int i = b + lane; i < e; i += 32) {
                        const int l = sidx[cur][i];
                        for (int k = 0; k < 3; ++k) {
                            const float c = centroid2(sbox[l], k);
                            cmin[k] = fminf(cmin[k], c);
                            cmax[k] = fmaxf(cmax[k], c);
                        }
                    }
                    float scale[3];
                    for (int k = 0; k < 3; ++k) {
                        cmin[k] = warp_min(cmin[k]);
                        cmax[k] = warp_max(cmax[k]);
                        scale[k] = sah_scale(cmin[k], cmax[k]);
                    }
                    sah_bins_clear(bins[warp], lane);
                    __syncwarp();
                    for (int i = b + lane; i < e; i += 32) sah_bins_add(bins[warp], sbox[sidx[cur][i]], cmin, scale);
                    __syncwarp();
                    float cost, whole[6];
                    int best;
                    sah_choose(bins[warp], lane, cost, best, whole);
                    if (lane == 31)
                        for (int c = 0; c < 6; ++c) node_box2[6 * node + c] = whole[c];
                    // all centroids equal (or one-sided bins), or the depth budget is used up: split the run in the middle
                    const bool median = !(cost < inf) || level + (32 - __clz(cnt - 1)) >= s_budget;
                    const int ax = best >> 5, sp = best & 31;
                    int nr = 0;
                    for (int base = b; base < e; base += 32) {
                        const int i = base + lane;
                        const bool valid = i < e;
                        const int l = valid ? sidx[cur][i] : 0;
                        bool go_left = false;
                        if (valid) {
                            if (median) go_left = (i - b) < cnt / 2;
                            else go_left = sah_bin(centroid2(sbox[l], ax), cmin[ax], scale[ax]) <= sp;
                        }
                        const unsigned ml = __ballot_sync(0xffffffffu, go_left), mr = __ballot_sync(0xffffffffu, valid && !go_left);
                        if (go_left) sidx[cur ^ 1][b + nl + __popc(ml & lt)] = (unsigned short)l;
                        else if (valid) sidx[cur ^ 1][e - 1 - (nr + __popc(mr & lt))] = (unsigned short)l;
                        nl += __popc(ml);
                        nr += __popc(mr);
                    }
                    __syncwarp();
                }
                if (lane == 0) emit(node, b, nl, e);
            }
            __syncthreads();
            // leaves that were not part of a task on this level keep their place in both index buffers only if they are
            // already emitted, so nothing has to be copied; flip the buffers
            if (tid == 0) q_n[cur] = 0;
            cur ^= 1;
            ++level;
            __syncthreads();
        }
    }
}

// one thread per leaf climbs; the second thread to reach a node computes its box.  NB boxes per entry: 1 = the canonical
// box (union over the shutter), 2 = the boxes at the two ends of the shutter (scenes with motion: the traversal nodes
// interpolate between them)
template <int NB>
__global__ void __launch_bounds__(TPB) k_refit(const uint64_t *__restrict__ keys, int n,
                                                const int *__restrict__ left, const int *__restrict__ right,
                                                const int *__restrict__ parent, const float *__restrict__ prim_box,
                                                float *node_box, int *visit)
{
    const int k = blockIdx.x * TPB + threadIdx.x;
    const int ni = n - 1;
    if (k >= n) return;
    int node = parent[ni + k];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&visit[node], 1) == 0) return;
        __threadfence();
        const int L = left[node], R = right[node];
        const volatile float *lb = L >= 0 ? node_box + 6 * NB * L : nullptr;
        const volatile float *rb = R >= 0 ? node_box + 6 * NB * R : nullptr;
        for (int e = 0; e < NB; ++e) {
            float l6[6], r6[6];
            for (int c = 0; c < 6; ++c) {
                l6[c] = L >= 0 ? lb[6 * e + c] : prim_box[6 * NB * (uint32_t)keys[~L] + 6 * e + c];
                r6[c] = R >= 0 ? rb[6 * e + c] : prim_box[6 * NB * (uint32_t)keys[~R] + 6 * e + c];
            }
            for (int c = 0; c < 3; ++c) {
                node_box[6 * NB * node + 6 * e + c] = fminf(l6[c], r6[c]);
                node_box[6 * NB * node + 6 * e + 3 + c] = fmaxf(l6[3 + c], r6[3 + c]);
            }
        }
        node = parent[node];
    }
}

// Refit of the traversal tree ABOVE the rebuilt subtrees, whose nodes got their boxes from k_sah_rebuild: one climber per
// subtree root, one per leaf that no subtree covers (a leaf, or a pair of leaves, hanging directly under a node of more
// than SAH_MAX leaves).  A scene that is one subtree needs no refit at all.
__global__ void __launch_bounds__(TPB) k_refit_upper(const uint64_t *__restrict__ keys, int n, const int *__restrict__ left,
                                                      const int *__restrict__ right, const int *__restrict__ parent,
                                                      const int *__restrict__ canon_parent, const int2 *__restrict__ range,
                                                      const float *__restrict__ prim_box, const int *__restrict__ roots,
                                                      const SahState *st, float *node_box, int *visit)
{
    const int k = blockIdx.x * TPB + threadIdx.x;
    const int ni = n - 1;
    int node;
    if (k < n) {
        // covered by a rebuilt subtree <=> some ancestor has 3 .. SAH_MAX leaves; sizes grow upwards, so it is the parent or,
        // under a parent of two leaves, the grandparent -- in the CANONICAL tree, whose ranges `range` holds (the parts of
        // the traversal tree that no subtree covers kept the canonical links)
        int p = canon_parent[ni + k];
        int size = range[p].y - range[p].x + 1;
        if (size == 2 && canon_parent[p] >= 0) {
            p = canon_parent[p];
            size = range[p].y - range[p].x + 1;
        }
        if (size >= 3 && size <= SAH_MAX) return;
        node = parent[ni + k];
    }
    else if (k - n < st->n_roots) node = parent[roots[k - n]];
    else return;
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&visit[node], 1) == 0) return;
        __threadfence();
        const int L = left[node], R = right[node];
        const volatile float *lb = L >= 0 ? node_box + 6 * L : nullptr;
        const volatile float *rb = R >= 0 ? node_box + 6 * R : nullptr;
        float l6[6], r6[6];
        for (int c = 0; c < 6; ++c) {
            l6[c] = L >= 0 ? lb[c] : prim_box[6 * (uint32_t)keys[~L] + c];
            r6[c] = R >= 0 ? rb[c] : prim_box[6 * (uint32_t)keys[~R] + c];
        }
        for (int c = 0; c < 3; ++c) {
            node_box[6 * node + c] = fminf(l6[c], r6[c]);
            node_box[6 * node + 3 + c] = fmaxf(l6[3 + c], r6[3 + c]);
        }
        node = parent[node];
    }
}

// traversal boxes are stored as centre + half extent (see box_hit): c +- h encloses [lo, hi] padded by `pad`
// (the roundings of c and of hi-c / c-lo are <= 2^-23 * magnitude, pad is 2^-20 * magnitude)
__device__ __forceinline__ void center_half(float lo, float hi, float pad, float &c, float &h)
{
    c = __fmul_rn(0.5f, __fadd_rn(lo, hi));
    h = __fadd_rn(fmaxf(__fsub_rn(hi, c), __fsub_rn(c, lo)), pad);
}

__device__ __forceinline__ int prim_type(int id, int ns, int nms, int nt)
{
    return id < ns ? PRIM_SPHERE : (id < ns + nms ? PRIM_MSPHERE : (id < ns + nms + nt ? PRIM_TRIANGLE : PRIM_MTRIANGLE));
}

// ---- 4-wide collapse of the canonical binary LBVH: the tree the render kernels traverse -----------------------------
// A wide node takes a binary node b and opens, twice, its internal child of largest surface area, which leaves up to
// four children (the greedy surface-area collapse of Wald et al. 2008 / Ylitie et al. 2017).  Wide nodes are created
// top-down through a work list: wq[i] = the binary node that roots wide node i, written by the thread that processed
// the parent (index taken from one atomic counter, so the array is in creation order: parents before children, roughly
// breadth-first).  One persistent grid drains the list: a warp draws 32 consecutive indices and polls their entries;
// an index whose entry never appears is past the end -- known once every primitive has been emitted as a leaf child
// (leaves_done == n), after which no node can be created.  The producer of an entry always holds a LOWER index, which
// was drawn earlier by a thread that is resident or finished, so the polling can not deadlock.
struct CollapseState {
    int n_alloc;     // wide nodes created so far (root included)
    int ticket;      // next index to hand out
    int leaves_done; // primitives emitted as leaf children
    int stuck;       // != 0: a warp gave up polling (a broken input tree would otherwise spin for ever): the build fails
};

__global__ void __launch_bounds__(TPB) k_collapse_init(int *__restrict__ wq, int n, CollapseState *st)
{
    const int i = blockIdx.x * TPB + threadIdx.x;
    if (i < n) wq[i] = i == 0 ? 0 : -1;
    if (i == 0) {
        st->n_alloc = 1;
        st->ticket = 0;
        st->leaves_done = 0;
        st->stuck = 0;
    }
}

// half extents travel as IEEE half precision (fp16) ROUNDED UP (a box may only grow: by < 2^-10 of its half extent, by at
// most 6e-8 below the smallest normal half, to +inf -- a slab that always passes -- above 65504); -inf (unused slot) is exact
__device__ __forceinline__ unsigned f16_up(float h) { return (unsigned)__half_as_ushort(__float2half_ru(h)); }
__device__ __forceinline__ float f16_pair_up(float lo, float hi) { return __uint_as_float(f16_up(lo) | (f16_up(hi) << 16)); }

__device__ __forceinline__ float box_area6(const float *b)
{
    return area_rn(__fsub_rn(b[3], b[0]), __fsub_rn(b[4], b[1]), __fsub_rn(b[5], b[2]));
}

__device__ __forceinline__ void collapse_one(int i, int b, const uint64_t *__restrict__ keys, int n, int ns, int nms, int nt,
                                             const int *__restrict__ left, const int *__restrict__ right,
                                             const float *__restrict__ prim_box, const float *__restrict__ node_box,
                                             const float *__restrict__ prim_box01, const float *__restrict__ node_box01,
                                             float pad, int *wq, CollapseState *st, float4 *__restrict__ wnodes)
{
    constexpr int WD = RRTB_WIDTH;
    int ch[WD];
    int nc;
    if (n == 1) { // degenerate tree: the only primitive is the root's only child
        ch[0] = ~0;
        nc = 1;
    }
    else {
        ch[0] = left[b];
        ch[1] = right[b];
        nc = 2;
        for (int rep = 0; rep < WD - 2; ++rep) {
            int bi = -1;
            float ba = -1.0f;
            for (int c = 0; c < nc; ++c)
                if (ch[c] >= 0) {
                    const float ar = box_area6(node_box + 6 * ch[c]);
                    if (ar > ba) {
                        ba = ar;
                        bi = c;
                    }
                }
            if (bi < 0) break;
            const int bb = ch[bi];
            ch[bi] = left[bb];
            ch[nc++] = right[bb];
        }
    }
    float cx[WD], cy[WD], cz[WD], hx[WD], hy[WD], hz[WD];
    float c1x[WD], c1y[WD], c1z[WD], h1x[WD], h1y[WD], h1z[WD]; // motion nodes: the box at the END of the shutter
    int ref[WD];
    int leaves = 0;
    const bool motion = prim_box01 != nullptr;
    for (int c = 0; c < WD; ++c) {
        if (c >= nc) { // unused slot: never hit
            cx[c] = cy[c] = cz[c] = c1x[c] = c1y[c] = c1z[c] = 0.f;
            hx[c] = hy[c] = hz[c] = h1x[c] = h1y[c] = h1z[c] = -__int_as_float(0x7f800000);
            ref[c] = TRAV_DONE;
            continue;
        }
        const float *bx;
        if (ch[c] >= 0) {
            const int j = atomicAdd(&st->n_alloc, 1);
            *(volatile int *)(wq + j) = ch[c];
            ref[c] = j;
            bx = motion ? node_box01 + 12 * ch[c] : node_box + 6 * ch[c];
        }
        else {
            const int slot = ~ch[c];
            const int id = (int)(uint32_t)keys[slot];
            ref[c] = ~((slot << 2) | prim_type(id, ns, nms, nt));
            bx = motion ? prim_box01 + 12 * id : prim_box + 6 * id;
            ++leaves;
        }
        center_half(bx[0], bx[3], pad, cx[c], hx[c]);
        center_half(bx[1], bx[4], pad, cy[c], hy[c]);
        center_half(bx[2], bx[5], pad, cz[c], hz[c]);
        if (motion) {
            center_half(bx[6], bx[9], pad, c1x[c], h1x[c]);
            center_half(bx[7], bx[10], pad, c1y[c], h1y[c]);
            center_half(bx[8], bx[11], pad, c1z[c], h1z[c]);
        }
    }
    if (motion) {
        // 160-byte motion node (rrtb_device.cuh "Motion node"): centres at both ends of the shutter, fp16 half extents
        // (rounded up) at both ends, refs; the traversal interpolates box(s) = (1 - s) box0 + s box1
        float4 *w = wnodes + RRTB_MOTION_NODE_F4 * (size_t)i;
        w[0] = make_float4(cx[0], cx[1], cx[2], cx[3]);
        w[1] = make_float4(cy[0], cy[1], cy[2], cy[3]);
        w[2] = make_float4(cz[0], cz[1], cz[2], cz[3]);
        w[3] = make_float4(c1x[0], c1x[1], c1x[2], c1x[3]);
        w[4] = make_float4(c1y[0], c1y[1], c1y[2], c1y[3]);
        w[5] = make_float4(c1z[0], c1z[1], c1z[2], c1z[3]);
        w[6] = make_float4(f16_pair_up(hx[0], hx[1]), f16_pair_up(hx[2], hx[3]), f16_pair_up(hy[0], hy[1]), f16_pair_up(hy[2], hy[3]));
        w[7] = make_float4(f16_pair_up(hz[0], hz[1]), f16_pair_up(hz[2], hz[3]), f16_pair_up(h1x[0], h1x[1]), f16_pair_up(h1x[2], h1x[3]));
        w[8] = make_float4(f16_pair_up(h1y[0], h1y[1]), f16_pair_up(h1y[2], h1y[3]), f16_pair_up(h1z[0], h1z[1]), f16_pair_up(h1z[2], h1z[3]));
        w[9] = make_float4(__int_as_float(ref[0]), __int_as_float(ref[1]), __int_as_float(ref[2]), __int_as_float(ref[3]));
    }
    else {
        // 96-byte node (rrtb_device.cuh "Traversal node"): float centres, fp16 half extents rounded up, refs
        float4 *w = wnodes + RRTB_NODE_F4 * (size_t)i;
        w[0] = make_float4(cx[0], cx[1], cx[2], cx[3]);
        w[1] = make_float4(cy[0], cy[1], cy[2], cy[3]);
        w[2] = make_float4(cz[0], cz[1], cz[2], cz[3]);
        w[3] = make_float4(f16_pair_up(hx[0], hx[1]), f16_pair_up(hx[2], hx[3]), f16_pair_up(hy[0], hy[1]), f16_pair_up(hy[2], hy[3]));
        w[4] = make_float4(f16_pair_up(hz[0], hz[1]), f16_pair_up(hz[2], hz[3]), __int_as_float(ref[0]), __int_as_float(ref[1]));
        w[5] = make_float4(__int_as_float(ref[2]), __int_as_float(ref[3]), 0.f, 0.f);
    }
    if (leaves) {
        __threadfence(); // the work-list entries written above are visible before the leaf count that ends the polling
        atomicAdd(&st->leaves_done, leaves);
    }
}

__global__ void __launch_bounds__(TPB) k_collapse4(const uint64_t *__restrict__ keys, int n, int ns, int nms, int nt,
                                                    const int *__restrict__ left, const int *__restrict__ right,
                                                    const float *__restrict__ prim_box, const float *__restrict__ node_box,
                                                    const float *__restrict__ prim_box01, const float *__restrict__ node_box01,
                                                    const BuildConsts *__restrict__ bc, int *wq, CollapseState *st,
                                                    float4 *__restrict__ wnodes)
{
    const unsigned lane = threadIdx.x & 31u;
    const float pad = bc->pad;
    const int max_nodes = max(n - 1, 1);
    while (true) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&st->ticket, 32);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= max_nodes) return;
        const int i = base + (int)lane;
        bool pending = i < max_nodes, past_end = false;
        unsigned spins = 0;
        while (__any_sync(0xffffffffu, pending)) {
            if (++spins > (1u << 24) || *(volatile int *)&st->stuck) { // never reached with a valid tree (tens of polls)
                st->stuck = 1;
                return;
            }
            if (pending) {
                int b = *(volatile int *)(wq + i);
                if (b < 0 && *(volatile int *)&st->leaves_done == n) {
                    __threadfence();
                    b = *(volatile int *)(wq + i); // look again: the entry may have landed just before the last leaf
                    if (b < 0) {
                        pending = false;
                        past_end = true;
                    }
                }
                if (b >= 0) {
                    collapse_one(i, b, keys, n, ns, nms, nt, left, right, prim_box, node_box, prim_box01, node_box01, pad, wq, st, wnodes);
                    pending = false;
                }
            }
        }
        if (__any_sync(0xffffffffu, past_end)) return; // every later index is past the end too
    }
}

__global__ void __launch_bounds__(TPB) k_flatten_leaves(const uint64_t *__restrict__ keys, int n,
                                                         const float4 *__restrict__ prim, const int2 *__restrict__ info,
                                                         const float4 *__restrict__ prim_ext, float4 *__restrict__ leaves,
                                                         int2 *__restrict__ leaf_info, float4 *__restrict__ leaf_ext)
{
    const int k = blockIdx.x * TPB + threadIdx.x;
    if (k >= n) return;
    const int id = (int)(uint32_t)keys[k];
    leaves[3 * k + 0] = prim[3 * id + 0];
    leaves[3 * k + 1] = prim[3 * id + 1];
    leaves[3 * k + 2] = prim[3 * id + 2];
    leaf_info[k] = info[id];
    if (prim_ext) { // scenes with moving triangles: their edge rates follow the record into leaf order
        leaf_ext[2 * k + 0] = prim_ext[2 * id + 0];
        leaf_ext[2 * k + 1] = prim_ext[2 * id + 1];
    }
}

// exposed to rrtb_api.cu (scene upload and rebuild): the raw struct arrays are staged in d_stage by the caller
int prepare_and_build(rrtb_ctx *ctx)
{
    const int n = ctx->n_prims;
    const int ns = ctx->n_spheres, nms = ctx->n_mspheres, nt = ctx->n_triangles;
    const int nb = (n + TPB - 1) / TPB;
    cudaStream_t st = ctx->stream;
    BuildConsts *bc = (BuildConsts *)(ctx->d_reduce + (size_t)nb * 7);
    const rrtb_sphere *d_sph = (const rrtb_sphere *)(ctx->d_stage + ctx->stage_off[0]);
    const rrtb_msphere *d_msph = (const rrtb_msphere *)(ctx->d_stage + ctx->stage_off[1]);
    const rrtb_triangle *d_tri = (const rrtb_triangle *)(ctx->d_stage + ctx->stage_off[2]);
    const rrtb_mtriangle *d_mtri = (const rrtb_mtriangle *)(ctx->d_stage + ctx->stage_off[3]);

    k_prepare<<<nb, TPB, 0, st>>>(d_sph, ns, d_msph, nms, d_tri, nt, d_mtri, ctx->n_mtriangles, ctx->cam.time0, ctx->cam.time1, ctx->d_prim,
                                  ctx->n_mtriangles > 0 ? ctx->d_prim_ext.get() : nullptr, ctx->d_prim_info, ctx->d_prim_box,
                                  ctx->motion ? ctx->d_prim_box01.get() : nullptr, ctx->d_reduce);
    float cam_mag = 0.f;
    for (int k = 0; k < 3; ++k) cam_mag = fmaxf(cam_mag, fabsf(ctx->cam.origin[k]) + ctx->cam.lens_radius);
    ctx->build_cam_mag = cam_mag;
    k_bounds<<<1, TPB, 0, st>>>(ctx->d_reduce, nb, cam_mag, bc);
    k_morton<<<nb, TPB, 0, st>>>(ctx->d_prim_box, n, bc, ctx->d_morton, ctx->d_keys);
    RRTB_CUDA(ctx, cudaGetLastError());

    // radix sort on the 30-bit code held in key bits 32..61
    const int n_seg = (n + SEG - 1) / SEG;
    const int sort_blocks = (n_seg + SORT_WARPS - 1) / SORT_WARPS;
    uint64_t *src = ctx->d_keys, *dst = ctx->d_keys_tmp;
    if (n <= SMALL_SORT) k_sort_small<<<1, 1024, 0, st>>>(ctx->d_keys, n);
    else for (int pass = 0; pass < 4; ++pass) {
        const int shift = 32 + 8 * pass;
        k_hist<<<sort_blocks, TPB, 0, st>>>(src, n, shift, n_seg, ctx->d_hist);
        const int hist_len = 256 * n_seg, scan_blocks = (hist_len + SCAN_CHUNK - 1) / SCAN_CHUNK;
        unsigned int *sums = ctx->d_hist + hist_len; // scan_blocks entries behind the histogram
        k_scan_sums<<<scan_blocks, TPB, 0, st>>>(ctx->d_hist, hist_len, sums);
        k_scan<<<1, 1024, 0, st>>>(sums, scan_blocks);
        k_scan_apply<<<scan_blocks, TPB, 0, st>>>(ctx->d_hist, hist_len, sums);
        k_scatter<<<sort_blocks, TPB, 0, st>>>(src, dst, n, shift, n_seg, ctx->d_hist);
        uint64_t *t = src;
        src = dst;
        dst = t;
    }
    RRTB_CUDA(ctx, cudaGetLastError());
    // 4 passes: result is back in d_keys (src == d_keys)

    // topology and boxes the traversal tree is collapsed from: the canonical LBVH, or its SAH-rebuilt copy
    const int *t_left = ctx->d_left, *t_right = ctx->d_right;
    const float *t_node_box = ctx->d_node_box;
    if (n > 1) {
        const int nbi = (n - 1 + TPB - 1) / TPB;
        k_karras<<<nbi, TPB, 0, st>>>(ctx->d_keys, n, ctx->d_left, ctx->d_right, ctx->d_parent, ctx->d_range);
        const int *t_parent = ctx->d_parent;
        RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_visit, 0, sizeof(int) * (size_t)(n - 1), st));
        if (n >= 3) { // SAH rebuild of every subtree of <= SAH_MAX leaves, for the traversal tree only
            SahState *ss = (SahState *)(ctx->d_collapse + 8);
            RRTB_CUDA(ctx, cudaMemsetAsync(ss, 0, sizeof(SahState), st));
            k_sah_select<<<(2 * n - 1 + TPB - 1) / TPB, TPB, 0, st>>>(n, ctx->d_left, ctx->d_right, ctx->d_parent, ctx->d_range, ctx->d_left2,
                                                                       ctx->d_right2, ctx->d_parent2, ctx->d_sah_roots, ss);
            const int max_roots = 2 * ((n + SAH_MAX - 1) / SAH_MAX) + 1; // maximal subtrees are disjoint and each parent covers > SAH_MAX leaves
            constexpr int SAH_BINS_BYTES = 3 * SAH_BINS * 7 * (int)sizeof(int); // per warp
            if (n <= 8 * SAH_MAX) {
                RRTB_CUDA(ctx, cudaFuncSetAttribute(k_sah_rebuild<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * SAH_BINS_BYTES));
                k_sah_rebuild<1024><<<min(max_roots, ctx->sm_count), 1024, 32 * SAH_BINS_BYTES, st>>>(
                    ctx->d_keys, n, ctx->d_range, ctx->d_prim_box, ctx->d_sah_roots, ctx->d_parent, ss, ctx->d_left2, ctx->d_right2, ctx->d_parent2,
                    ctx->d_node_box2);
            }
            else
                k_sah_rebuild<256><<<min(max_roots, ctx->sm_count * 4), 256, 8 * SAH_BINS_BYTES, st>>>(
                    ctx->d_keys, n, ctx->d_range, ctx->d_prim_box, ctx->d_sah_roots, ctx->d_parent, ss, ctx->d_left2, ctx->d_right2, ctx->d_parent2,
                    ctx->d_node_box2);
            k_refit_upper<<<(n + max_roots + TPB - 1) / TPB, TPB, 0, st>>>(ctx->d_keys, n, ctx->d_left2, ctx->d_right2, ctx->d_parent2, ctx->d_parent, ctx->d_range,
                                                                            ctx->d_prim_box, ctx->d_sah_roots, ss, ctx->d_node_box2, ctx->d_visit);
            t_left = ctx->d_left2;
            t_right = ctx->d_right2;
            t_parent = ctx->d_parent2;
            t_node_box = ctx->d_node_box2;
            // the boxes of the canonical tree are needed by rrtb_bvh_download only: refit_canonical() on demand
            ctx->canonical_boxes = false;
        }
        else {
            k_refit<1><<<nb, TPB, 0, st>>>(ctx->d_keys, n, ctx->d_left, ctx->d_right, ctx->d_parent, ctx->d_prim_box,
                                           ctx->d_node_box, ctx->d_visit);
            ctx->canonical_boxes = true;
        }
        if (ctx->motion) { // boxes at the two ends of the shutter, for the interpolating traversal nodes
            RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_visit, 0, sizeof(int) * (size_t)(n - 1), st));
            k_refit<2><<<nb, TPB, 0, st>>>(ctx->d_keys, n, t_left, t_right, t_parent, ctx->d_prim_box01,
                                           ctx->d_node_box01, ctx->d_visit);
        }
    }
    else {
        int m1 = -1;
        RRTB_CUDA(ctx, cudaMemcpyAsync(ctx->d_parent, &m1, sizeof(int), cudaMemcpyHostToDevice, st));
    }
    CollapseState *cs = (CollapseState *)ctx->d_collapse.get();
    k_collapse_init<<<nb, TPB, 0, st>>>(ctx->d_wq, n, cs);
    const int want_blocks = (max(n - 1, 1) + TPB - 1) / TPB;
    k_collapse4<<<min(want_blocks, ctx->sm_count * 4), TPB, 0, st>>>(ctx->d_keys, n, ns, nms, nt, t_left, t_right,
                                                                     ctx->d_prim_box, t_node_box, ctx->motion ? ctx->d_prim_box01.get() : nullptr,
                                                                     ctx->motion ? ctx->d_node_box01.get() : nullptr, bc, ctx->d_wq, cs, ctx->d_wnodes);
    const bool has_ext = ctx->n_mtriangles > 0;
    k_flatten_leaves<<<nb, TPB, 0, st>>>(ctx->d_keys, n, ctx->d_prim, ctx->d_prim_info, has_ext ? ctx->d_prim_ext.get() : nullptr, ctx->d_leaves,
                                         ctx->d_leaf_info, has_ext ? ctx->d_leaf_ext.get() : nullptr);
    RRTB_CUDA(ctx, cudaGetLastError());
    return RRTB_OK;
}

// Boxes of the canonical LBVH (rrtb_bvh_download; the traversal tree has its own): refit once, when first asked for.
int refit_canonical(rrtb_ctx *ctx)
{
    const int n = ctx->n_prims;
    if (ctx->canonical_boxes || n < 2) return RRTB_OK;
    cudaStream_t st = ctx->stream;
    RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_visit, 0, sizeof(int) * (size_t)(n - 1), st));
    k_refit<1><<<(n + TPB - 1) / TPB, TPB, 0, st>>>(ctx->d_keys, n, ctx->d_left, ctx->d_right, ctx->d_parent, ctx->d_prim_box,
                                                    ctx->d_node_box, ctx->d_visit);
    RRTB_CUDA(ctx, cudaGetLastError());
    RRTB_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->canonical_boxes = true;
    return RRTB_OK;
}

} // namespace rrtb
