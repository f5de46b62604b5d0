// rrtb_path.cuh -- the PATH POLICY: what the render kernels and the test hooks need to know about an integrator.
//
// PathF32 is the float integrator (rrtb_device.cuh, the headline build), PathF64 the double integrator of
// rrtb_device_f64.cuh (SURVEY 8f1).  A policy only names types and forwards to the device functions of its
// integrator, whose arithmetic stays separate (each is bit-exact against its own oracle); the closest-hit queries
// below, the lane and pool kernels (rrtb_render.cu, rrtb_render_pool.cuh) and the hooks are written once over it.
#pragma once
#include <type_traits>

#include "rrtb_device_f64.cuh"

#ifndef RRTB_POOL
#define RRTB_POOL 96 // float integrator: path slots per warp (64 / 80 / 112 measured slower, profiles/README.md)
#endif

namespace rrtb {

struct PathF32 { // the float integrator (rrtb_device.cuh)
    typedef float real;
    typedef Ray RayT;
    typedef Hit HitT;
    typedef HitRecord RecT;
    static constexpr int POOL = RRTB_POOL;  // pool scheduler: path slots per warp
    static constexpr int BLOCKS_PER_SM = 4; // 64 registers
    static __device__ __forceinline__ RayPre pre(const Ray &r) { return ray_pre(r); }
    static __device__ __forceinline__ float inf() { return __int_as_float(0x7f800000); }
    static __device__ __forceinline__ float t_min_f(float t_min) { return t_min; }
    static __device__ __forceinline__ float t_max_f(const Hit &h) { return h.t; }
    static __device__ __forceinline__ Hit make_hit(float t, int ref)
    {
        Hit h;
        h.t = t;
        h.ref = ref;
        h.obj = -1;
        return h;
    }
    template <bool COUNT, bool MTRI>
    static __device__ __forceinline__ void leaf(const float4 *__restrict__ leaves, const LeafAux info, int slot, int type,
                                                const Ray &r, const RayPre &p, float t_min, Hit &best, TravCounters &tc)
    {
        leaf_test<COUNT, MTRI>(leaves, info, slot, type, r, p, t_min, best, tc);
    }
    template <bool MTRI>
    static __device__ __forceinline__ HitRecord record(const float4 *__restrict__ leaves, const LeafAux info,
                                                       const Ray &r, const Hit &h)
    {
        return hit_record<MTRI>(leaves, info, r, h);
    }
    template <bool LIGHTS = false>
    static __device__ __forceinline__ bool bounce(int mtype, float4 m, const Ray &r, const HitRecord &rec, uint4 rnd, float &dx,
                                                  float &dy, float &dz, float &ar, float &ag, float &ab)
    {
        return scatter<LIGHTS>(mtype, m, r, rec, rnd, dx, dy, dz, ar, ag, ab);
    }
    static __device__ __forceinline__ float mul(float x, float y) { return x * y; }
    // sky x throughput -> fixed point (rrt.cu:68-75), clamped to fixed_clamp(spp)
    static __device__ __forceinline__ void sky_fixed(const Ray &r, float tr, float tg, float tb, float clamp, unsigned long long &fr,
                                                     unsigned long long &fg, unsigned long long &fb)
    {
        float cr, cg, cb;
        sky(r, cr, cg, cb);
        fr = to_fixed(tr * cr, clamp);
        fg = to_fixed(tg * cg, clamp);
        fb = to_fixed(tb * cb, clamp);
    }
    // throughput x a constant radiance -> fixed point: the emitted term (Le of a RRTB_DIFFUSE_LIGHT hit, material
    // albedo) and the background term (a segment that leaves a scene with a background), plain float products as above
    static __device__ __forceinline__ void const_fixed(float tr, float tg, float tb, float lr, float lg, float lb, float clamp,
                                                       unsigned long long &fr, unsigned long long &fg, unsigned long long &fb)
    {
        fr = to_fixed(tr * lr, clamp);
        fg = to_fixed(tg * lg, clamp);
        fb = to_fixed(tb * lb, clamp);
    }
    static __device__ __forceinline__ Ray camera(const DeviceCamera &cam, int W, int H, int i, int j, int sample, uint2 key)
    {
        return camera_ray(cam, W, H, i, j, sample, key);
    }
    // first-hit AOVs: the clamped albedo of a hit and the distance to it
    static __device__ __forceinline__ void albedo(int mtype, float4 m, float &r, float &g, float &b) { aov_albedo(mtype, m, r, g, b); }
    static __device__ __forceinline__ float distance(const Ray &r, float t) { return ray_distance(r, t); }
};

struct PathF64 { // the double integrator (rrtb_device_f64.cuh); bit-exact against oracle/rrt_oracle_f64.c
    typedef double real;
    typedef RayD RayT;
    typedef HitD HitT;
    typedef HitRecordD RecT;
    // measured on final.txt / synthetic (ms at 64 / 8 spp): POOL x blocks 96x2 15.7 / 44.1, 128x2 17.6 / 48.6,
    // 80x3 15.2 / 38.0, 72x3 14.1 / 36.7, 64x3 14.0 / 37.4, 56x3 14.6 / 40.7, 48x3 15.3 / 45.2, 48x4 15.5 / 44.2
    static constexpr int POOL = 64;
    static constexpr int BLOCKS_PER_SM = 3; // 80 registers, 55 KB of slots per block
    // the slab tests run in float on the float view of the ray (ray_pre_d); the running closest distance is rounded
    // UP and t_min DOWN when they enter them
    static __device__ __forceinline__ RayPre pre(const RayD &r) { return ray_pre_d(r); }
    static __device__ __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000ll); }
    static __device__ __forceinline__ float t_min_f(double t_min) { return __double2float_rd(t_min); }
    static __device__ __forceinline__ float t_max_f(const HitD &h) { return __double2float_ru(h.t); }
    static __device__ __forceinline__ HitD make_hit(double t, int ref)
    {
        HitD h;
        h.t = t;
        h.ref = ref;
        return h;
    }
    template <bool COUNT, bool MTRI>
    static __device__ __forceinline__ void leaf(const float4 *__restrict__ leaves, const LeafAux info, int slot, int type,
                                                const RayD &r, const RayPre &, double t_min, HitD &best, TravCounters &tc)
    {
        leaf_test_d<COUNT>(leaves, info, slot, type, r, t_min, best, tc);
    }
    template <bool MTRI>
    static __device__ __forceinline__ HitRecordD record(const float4 *__restrict__ leaves, const LeafAux info,
                                                        const RayD &r, const HitD &h)
    {
        return hit_record_d(leaves, info, r, h);
    }
    template <bool LIGHTS = false>
    static __device__ __forceinline__ bool bounce(int mtype, float4 m, const RayD &r, const HitRecordD &rec, uint4 rnd, double &dx,
                                                  double &dy, double &dz, double &ar, double &ag, double &ab)
    {
        return scatter_d<LIGHTS>(mtype, m, r, rec, rnd, dx, dy, dz, ar, ag, ab);
    }
    static __device__ __forceinline__ double mul(double x, double y) { return __dmul_rn(x, y); }
    static __device__ __forceinline__ void sky_fixed(const RayD &r, double tr, double tg, double tb, float clamp, unsigned long long &fr,
                                                     unsigned long long &fg, unsigned long long &fb)
    {
        double lr, lg, lb;
        sky_d(r, tr, tg, tb, lr, lg, lb);
        fr = to_fixed_d(lr, clamp);
        fg = to_fixed_d(lg, clamp);
        fb = to_fixed_d(lb, clamp);
    }
    // the emitted and background terms: __dmul_rn(throughput, (double)L), as oracle/rrt_oracle_f64.c
    static __device__ __forceinline__ void const_fixed(double tr, double tg, double tb, float lr, float lg, float lb, float clamp,
                                                       unsigned long long &fr, unsigned long long &fg, unsigned long long &fb)
    {
        fr = to_fixed_d(__dmul_rn(tr, (double)lr), clamp);
        fg = to_fixed_d(__dmul_rn(tg, (double)lg), clamp);
        fb = to_fixed_d(__dmul_rn(tb, (double)lb), clamp);
    }
    static __device__ __forceinline__ RayD camera(const DeviceCamera &cam, int W, int H, int i, int j, int sample, uint2 key)
    {
        return camera_ray_d(cam, W, H, i, j, sample, key);
    }
    // the albedo is clamped in float and widened: exact, and the same as clamping the widened value
    static __device__ __forceinline__ void albedo(int mtype, float4 m, double &r, double &g, double &b)
    {
        float fr, fg, fb;
        aov_albedo(mtype, m, fr, fg, fb);
        r = fr;
        g = fg;
        b = fb;
    }
    static __device__ __forceinline__ double distance(const RayD &r, double t) { return ray_distance_d(r, t); }
};

template <typename real>
using PathOf = typename std::conditional<std::is_same<real, double>::value, PathF64, PathF32>::type;

// the leaf reference `cur` (rrtb_device.cuh "closest hit"): exact primitive test, then pop
template <class P, bool COUNT, bool MTRI>
__device__ __forceinline__ void leaf_step(const float4 *__restrict__ leaves, const LeafAux info, const typename P::RayT &r,
                                          const RayPre &p, typename P::real t_min, typename P::HitT &best, int &cur, TravSp &sp,
                                          const int *stk, TravCounters &cnt)
{
    P::template leaf<COUNT, MTRI>(leaves, info, (~cur) >> 2, (~cur) & 3, r, p, t_min, best, cnt);
    trav_pop(cur, sp, stk);
}

// ---- closest hit: flat scan (hittable_list.h:95-117) ------------------------------------------------------
template <class P, bool COUNT>
__device__ __forceinline__ typename P::HitT closest_scan(const DeviceScene &s, const typename P::RayT &r, typename P::real t_min,
                                                         TravCounters &cnt)
{
    typename P::HitT best = P::make_hit(P::inf(), -1);
    const RayPre p = P::pre(r);
    const int n0 = s.n_spheres, n1 = n0 + s.n_mspheres, n2 = n1 + s.n_triangles, n = s.n_prims;
    for (int k = 0; k < n; ++k) {
        int type = k < n0 ? PRIM_SPHERE : (k < n1 ? PRIM_MSPHERE : (k < n2 ? PRIM_TRIANGLE : PRIM_MTRIANGLE));
        P::template leaf<COUNT, true>(s.flat_leaves, LeafAux{s.flat_info, s.flat_ext}, k, type, r, p, t_min, best, cnt);
    }
    return best;
}

// ---- closest hit: traversal of the 4-wide tree (bvh_node::hit, bvh.h:167-175), one ray to the end --------------
template <class P, bool COUNT>
__device__ __forceinline__ typename P::HitT closest_bvh(const DeviceScene &s, const typename P::RayT &r, typename P::real t_min,
                                                        TravCounters &cnt)
{
    typename P::HitT best = P::make_hit(P::inf(), -1);
    const RayPre p = P::pre(r);
    const LeafAux info = {s.leaf_info, s.leaf_ext};
    int stack[RRTB_STACK];
    TravSp sp;
    int cur;
    trav_begin(cur, sp, stack);
    if (s.motion) { // interpolating nodes: where the ray's time lies in the shutter
        RayPre pm = p;
        pm.s = ((float)r.tm - s.shutter_open) * s.shutter_inv;
        while (cur != TRAV_DONE) {
            if (cur >= 0) wide_step<COUNT, true>(s.wnodes, pm, P::t_min_f(t_min), P::t_max_f(best), cur, sp, stack, cnt);
            else leaf_step<P, COUNT, true>(s.leaves, info, r, p, t_min, best, cur, sp, stack, cnt);
        }
        return best;
    }
    while (cur != TRAV_DONE) {
        if (cur >= 0) wide_step<COUNT>(s.wnodes, p, P::t_min_f(t_min), P::t_max_f(best), cur, sp, stack, cnt);
        else leaf_step<P, COUNT, true>(s.leaves, info, r, p, t_min, best, cur, sp, stack, cnt);
    }
    return best;
}

} // namespace rrtb
