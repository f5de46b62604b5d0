// rrtb_device_f64.cuh -- the DOUBLE-precision integrator (SURVEY 8f1): what the reference's `rrtd` build computes
// (FP_T = double, rtweekend.h:20-28, Makefile:36-37) over the float-rounded scene the C ABI carries.
//
// Rays, hit points, normals, scattering and throughput are double; the Philox streams, the direct samplers, the
// LBVH and the tie rule are the float integrator's.  The slab tests stay in float on the float-rounded ray: the
// node boxes are padded by 2^-20 * scene magnitude, 16x the rounding of the ray, so they remain conservative,
// and exactness lives in the double leaf tests.
//
// EVERY arithmetic operation below is an explicit round-to-nearest intrinsic in the order oracle/rrt_oracle_f64.c
// performs it: IEEE double add/mul/fma/div/sqrt are correctly rounded on both sides, so the whole integrator --
// not only the intersection code -- is BIT-EXACT against the CPU oracle (tests/test_gpu_f64.py compares the
// fixed-point framebuffers for equality).
#pragma once
#include "rrtb_device.cuh"

namespace rrtb {

struct RayD {
    double ox, oy, oz, dx, dy, dz, tm;
};

struct HitD {
    double t;
    int ref; // (slot << 2) | type, -1 = miss
};

struct HitRecordD {
    double px, py, pz, nx, ny, nz;
    bool front;
    int obj, mat;
};

__device__ __forceinline__ double u01d(uint32_t x) { return __dmul_rn((double)(x >> 8), 5.9604644775390625e-08); }

__device__ __forceinline__ double ddot3(double ax, double ay, double az, double bx, double by, double bz)
{
    return __fma_rn(az, bz, __fma_rn(ay, by, __dmul_rn(ax, bx)));
}

// the float integrator's quadrant-exact polynomial evaluated in double (sampling needs no more accuracy)
__device__ __forceinline__ void sincos2pi_d(double u, double &co, double &si)
{
    double x = __dadd_rn(u, -0.5);
    double qf = rint(__dmul_rn(x, 4.0));
    double r = __fma_rn(qf, -0.25, x);
    double a = __dmul_rn(r, 6.283185307179586);
    double a2 = __dmul_rn(a, a);
    double sp = __fma_rn(a2, -1.9515295891e-4, 8.3321608736e-3);
    sp = __fma_rn(a2, sp, -1.6666654611e-1);
    double sn = __fma_rn(__dmul_rn(a, a2), sp, a);
    double cp = __fma_rn(a2, 2.443315711809948e-5, -1.388731625493765e-3);
    cp = __fma_rn(a2, cp, 4.166664568298827e-2);
    cp = __fma_rn(a2, cp, -0.5);
    double cs = __fma_rn(a2, cp, 1.0);
    int q = (int)qf & 3;
    co = (q & 1) ? sn : cs;
    si = (q & 1) ? cs : sn;
    if (q == 1 || q == 2) co = -co;
    if (q >= 2) si = -si;
}

// ---- primary rays: rrt.cu:112-114 + camera.h:31-38 in double ----------------------------------------------
__device__ __forceinline__ RayD camera_ray_d(const DeviceCamera &cam, int W, int H, int i, int j, int sample, uint2 key)
{
    const int pixel = j * W + i;
    uint4 b0 = philox4x32_10(make_uint4((uint32_t)pixel, (uint32_t)sample, 0u, 0u), key);
    double u = __ddiv_rn(__dadd_rn((double)i, u01d(b0.x)), (double)(W - 1));
    double v = __ddiv_rn(__dadd_rn((double)j, u01d(b0.y)), (double)(H - 1));
    double of[3] = {0.0, 0.0, 0.0};
    if (cam.lens_radius > 0.0f) {
        double r = __dmul_rn(__dsqrt_rn(u01d(b0.z)), (double)cam.lens_radius);
        double c, s;
        sincos2pi_d(u01d(b0.w), c, s);
        double rdx = __dmul_rn(r, c), rdy = __dmul_rn(r, s);
#pragma unroll
        for (int k = 0; k < 3; ++k) of[k] = __fma_rn((double)cam.v[k], rdy, __dmul_rn((double)cam.u[k], rdx));
    }
    double o[3], d[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double org = (double)cam.origin[k];
        o[k] = __dadd_rn(org, of[k]);
        double at = __fma_rn(v, (double)cam.vertical[k], __fma_rn(u, (double)cam.horizontal[k], (double)cam.llc[k]));
        d[k] = __dsub_rn(__dsub_rn(at, org), of[k]);
    }
    RayD r;
    r.ox = o[0]; r.oy = o[1]; r.oz = o[2];
    r.dx = d[0]; r.dy = d[1]; r.dz = d[2];
    r.tm = (double)cam.time0;
    if (cam.time0 != cam.time1) {
        uint4 b1 = philox4x32_10(make_uint4((uint32_t)pixel, (uint32_t)sample, 1u, 0u), key);
        r.tm = __fma_rn(__dsub_rn((double)cam.time1, (double)cam.time0), u01d(b1.x), (double)cam.time0);
    }
    return r;
}

// the float view of a double ray that drives the (conservative) slab tests
__device__ __forceinline__ RayPre ray_pre_d(const RayD &r)
{
    Ray f;
    f.ox = __double2float_rn(r.ox); f.oy = __double2float_rn(r.oy); f.oz = __double2float_rn(r.oz);
    f.dx = __double2float_rn(r.dx); f.dy = __double2float_rn(r.dy); f.dz = __double2float_rn(r.dz);
    f.tm = 0.f;
    return ray_pre(f);
}

// ---- primitive tests ------------------------------------------------------------------------------------
// sphere.h:33-58 in double; the roots through the cancellation-free pair q/a, c/q
__device__ __forceinline__ bool sphere_test_d(const RayD &r, double cx, double cy, double cz, double rad, double t_min,
                                              double t_max, double &t_out)
{
    double ocx = __dsub_rn(r.ox, cx), ocy = __dsub_rn(r.oy, cy), ocz = __dsub_rn(r.oz, cz);
    double a = ddot3(r.dx, r.dy, r.dz, r.dx, r.dy, r.dz);
    double hb = ddot3(ocx, ocy, ocz, r.dx, r.dy, r.dz);
    double cc = __fma_rn(-rad, rad, ddot3(ocx, ocy, ocz, ocx, ocy, ocz));
    double disc = __fma_rn(-a, cc, __dmul_rn(hb, hb));
    if (disc < 0.0) return false;
    double sq = __dsqrt_rn(disc);
    double q = -__dadd_rn(hb, copysign(sq, hb));
    double r0 = __ddiv_rn(q, a), r1 = __ddiv_rn(cc, q);
    double tn = fmin(r0, r1), tf = fmax(r0, r1);
    double root = tn;
    if (!(root >= t_min && root <= t_max)) {
        root = tf;
        if (!(root >= t_min && root <= t_max)) return false;
    }
    t_out = root;
    return true;
}

// moving_sphere.h:27-30 on the leaf record a = (c0, r), b = (c1 - c0, t0), c = (t1 - t0, ...)
__device__ __forceinline__ void msphere_center_d(float4 a, float4 b, float4 c, double time, double &cx, double &cy,
                                                 double &cz)
{
    double k = __ddiv_rn(__dsub_rn(time, (double)b.w), (double)c.x);
    cx = __fma_rn(k, (double)b.x, (double)a.x);
    cy = __fma_rn(k, (double)b.y, (double)a.y);
    cz = __fma_rn(k, (double)b.z, (double)a.z);
}

// triangle.h:35-75 in double
__device__ __forceinline__ bool triangle_test_d(const RayD &r, double v0x, double v0y, double v0z, float4 B, float4 C,
                                                double t_min, double t_max, double &t_out)
{
    const double EPS = 1e-7;
    double e1x = B.x, e1y = B.y, e1z = B.z, e2x = C.x, e2y = C.y, e2z = C.z;
    double hx = dcross(r.dy, e2z, r.dz, e2y), hy = dcross(r.dz, e2x, r.dx, e2z), hz = dcross(r.dx, e2y, r.dy, e2x);
    double det = ddot3(e1x, e1y, e1z, hx, hy, hz);
    if (det > -EPS && det < EPS) return false;
    double sx = __dsub_rn(r.ox, v0x), sy = __dsub_rn(r.oy, v0y), sz = __dsub_rn(r.oz, v0z);
    double un = ddot3(sx, sy, sz, hx, hy, hz);
    double qx = dcross(sy, e1z, sz, e1y), qy = dcross(sz, e1x, sx, e1z), qz = dcross(sx, e1y, sy, e1x);
    double vn = ddot3(r.dx, r.dy, r.dz, qx, qy, qz);
    if (det > 0.0) {
        if (un < 0.0 || un > det || vn < 0.0 || __dadd_rn(un, vn) > det) return false;
    }
    else {
        if (un > 0.0 || un < det || vn > 0.0 || __dadd_rn(un, vn) < det) return false;
    }
    double t = __ddiv_rn(ddot3(e2x, e2y, e2z, qx, qy, qz), det);
    if (t > EPS && t > t_min && t <= t_max) { // t == t_max: exact tie, settled by the tie rule
        t_out = t;
        return true;
    }
    return false;
}

template <bool COUNT>
__device__ __forceinline__ void leaf_test_d(const float4 *__restrict__ leaves, const LeafAux info, int slot,
                                            int type, const RayD &r, double t_min, HitD &best, TravCounters &cnt)
{
    if (COUNT) {
        if (type == PRIM_SPHERE) ++cnt.sph;
        else if (type == PRIM_MSPHERE) ++cnt.msph;
        else ++cnt.tri;
    }
    const float4 *rec = leaves + (size_t)(unsigned)slot * 3u; // one IMAD.WIDE (slot * 48 + base)
    double t;
    bool h;
    if (type == PRIM_SPHERE) { // centre and radius as doubles in the second and third float4 (k_prepare)
        const float4 b = __ldg(rec + 1), c = __ldg(rec + 2);
        h = sphere_test_d(r, __hiloint2double(__float_as_int(b.y), __float_as_int(b.x)),
                          __hiloint2double(__float_as_int(b.w), __float_as_int(b.z)),
                          __hiloint2double(__float_as_int(c.y), __float_as_int(c.x)),
                          __hiloint2double(__float_as_int(c.w), __float_as_int(c.z)), t_min, best.t, t);
    }
    else if (type == PRIM_MSPHERE) {
        float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
        double cx, cy, cz;
        msphere_center_d(a, b, c, r.tm, cx, cy, cz);
        h = sphere_test_d(r, cx, cy, cz, (double)a.w, t_min, best.t, t);
    }
    else {
        float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
        double v0x = a.x, v0y = a.y, v0z = a.z;
        if (type == PRIM_MTRIANGLE) {
            v0x = __fma_rn((double)a.w, r.tm, v0x);
            v0y = __fma_rn((double)b.w, r.tm, v0y);
            v0z = __fma_rn((double)c.w, r.tm, v0z);
            mtri_edges(info.ext, slot, __double2float_rn(r.tm), b, c); // the float edges of the pose at the float view of the time
        }
        h = triangle_test_d(r, v0x, v0y, v0z, b, c, t_min, best.t, t);
    }
    if (!h) return;
    if (best.ref >= 0 && t == best.t) { // exact tie: the float integrator's rule, by object id
        int obj = __ldg(&info.info[slot]).x;
        int bobj = __ldg(&info.info[best.ref >> 2]).x;
        if (!candidate_wins(0.f, type, obj, 0.f, best.ref & 3, bobj)) return;
    }
    best.t = t;
    best.ref = (slot << 2) | type;
}

// ---- hit record: sphere.h:51-55, moving_sphere.h:51-55, triangle.h:62-66, hittable.h:16-20 ---------------
__device__ __forceinline__ HitRecordD hit_record_d(const float4 *__restrict__ leaves, const LeafAux info,
                                                   const RayD &r, const HitD &h)
{
    HitRecordD rec;
    int slot = h.ref >> 2, type = h.ref & 3;
    rec.px = __fma_rn(h.t, r.dx, r.ox);
    rec.py = __fma_rn(h.t, r.dy, r.oy);
    rec.pz = __fma_rn(h.t, r.dz, r.oz);
    float4 a = __ldg(leaves + 3 * slot);
    if (type == PRIM_TRIANGLE) { // the stored unit face normal (float, triangle.h:9-15)
        float4 b = __ldg(leaves + 3 * slot + 1), c = __ldg(leaves + 3 * slot + 2);
        rec.nx = (double)a.w;
        rec.ny = (double)b.w;
        rec.nz = (double)c.w;
    }
    else if (type == PRIM_MTRIANGLE) {
        float4 b = __ldg(leaves + 3 * slot + 1), c = __ldg(leaves + 3 * slot + 2);
        mtri_edges(info.ext, slot, __double2float_rn(r.tm), b, c);
        float3 n = triangle_unit_normal_cold(b, c);
        rec.nx = (double)n.x;
        rec.ny = (double)n.y;
        rec.nz = (double)n.z;
    }
    else {
        double cx = a.x, cy = a.y, cz = a.z;
        if (type == PRIM_MSPHERE) {
            float4 b = __ldg(leaves + 3 * slot + 1), c = __ldg(leaves + 3 * slot + 2);
            msphere_center_d(a, b, c, r.tm, cx, cy, cz);
        }
        double inv = __ddiv_rn(1.0, (double)a.w);
        rec.nx = __dmul_rn(inv, __dsub_rn(rec.px, cx));
        rec.ny = __dmul_rn(inv, __dsub_rn(rec.py, cy));
        rec.nz = __dmul_rn(inv, __dsub_rn(rec.pz, cz));
    }
    double dn = __dadd_rn(__dadd_rn(__dmul_rn(r.dx, rec.nx), __dmul_rn(r.dy, rec.ny)), __dmul_rn(r.dz, rec.nz));
    rec.front = dn < 0.0;
    if (!rec.front) {
        rec.nx = -rec.nx;
        rec.ny = -rec.ny;
        rec.nz = -rec.nz;
    }
    int2 inf = __ldg(&info.info[slot]);
    rec.obj = inf.x;
    rec.mat = inf.y;
    return rec;
}

// ---- materials: material.h:21-32,48-57,76-109 + vec3.h:156-164 in double, one Philox block per bounce -----
__device__ __forceinline__ void sample_unit_sphere_d(double x0, double x1, double &ux, double &uy, double &uz)
{
    double z = __fma_rn(-2.0, x0, 1.0);
    double rr = __dsqrt_rn(fmax(0.0, __fma_rn(-z, z, 1.0)));
    double c, s;
    sincos2pi_d(x1, c, s);
    ux = __dmul_rn(rr, c);
    uy = __dmul_rn(rr, s);
    uz = z;
}

__device__ __forceinline__ bool scatter_d(int mtype, float4 m, const RayD &r, const HitRecordD &rec, uint4 rnd, double &dx,
                                          double &dy, double &dz, double &ar, double &ag, double &ab)
{
    const double nx = rec.nx, ny = rec.ny, nz = rec.nz;
    if (mtype == 0) {
        double ux, uy, uz;
        sample_unit_sphere_d(u01d(rnd.x), u01d(rnd.y), ux, uy, uz);
        dx = __dadd_rn(nx, ux);
        dy = __dadd_rn(ny, uy);
        dz = __dadd_rn(nz, uz);
        if (fabs(dx) < 1e-8 && fabs(dy) < 1e-8 && fabs(dz) < 1e-8) {
            dx = nx;
            dy = ny;
            dz = nz;
        }
        ar = m.x;
        ag = m.y;
        ab = m.z;
        return true;
    }
    double inv = __ddiv_rn(1.0, __dsqrt_rn(ddot3(r.dx, r.dy, r.dz, r.dx, r.dy, r.dz)));
    double udx = __dmul_rn(inv, r.dx), udy = __dmul_rn(inv, r.dy), udz = __dmul_rn(inv, r.dz);
    double dn = ddot3(udx, udy, udz, nx, ny, nz);
    if (mtype == 1) {
        double k = __dmul_rn(-2.0, dn);
        dx = __fma_rn(k, nx, udx);
        dy = __fma_rn(k, ny, udy);
        dz = __fma_rn(k, nz, udz);
        double fuzz = m.w < 1.0f ? (double)m.w : 1.0;
        if (fuzz > 0.0) {
            double ux, uy, uz;
            sample_unit_sphere_d(u01d(rnd.x), u01d(rnd.y), ux, uy, uz);
            double ra = u01d(rnd.z);
            double rb = __dmul_rn((double)(rnd.w >> 16), 1.52587890625e-05);
            double rc = __dmul_rn((double)(rnd.w & 0xFFFFu), 1.52587890625e-05);
            double rad = __dmul_rn(fmax(ra, fmax(rb, rc)), fuzz);
            dx = __fma_rn(rad, ux, dx);
            dy = __fma_rn(rad, uy, dy);
            dz = __fma_rn(rad, uz, dz);
        }
        ar = m.x;
        ag = m.y;
        ab = m.z;
        return ddot3(dx, dy, dz, nx, ny, nz) > 0.0;
    }
    double ir = m.w;
    double eta = rec.front ? __ddiv_rn(1.0, ir) : ir;
    double cos_t = fmin(-dn, 1.0);
    double sin_t = __dsqrt_rn(fmax(0.0, __fma_rn(-cos_t, cos_t, 1.0)));
    bool cannot = __dmul_rn(eta, sin_t) > 1.0;
    double r0 = __ddiv_rn(__dsub_rn(1.0, eta), __dadd_rn(1.0, eta));
    r0 = __dmul_rn(r0, r0);
    double om = __dsub_rn(1.0, cos_t), om2 = __dmul_rn(om, om);
    double refl_p = __fma_rn(__dsub_rn(1.0, r0), __dmul_rn(__dmul_rn(om2, om2), om), r0);
    if (cannot || refl_p > u01d(rnd.x)) {
        double k = __dmul_rn(-2.0, dn);
        dx = __fma_rn(k, nx, udx);
        dy = __fma_rn(k, ny, udy);
        dz = __fma_rn(k, nz, udz);
    }
    else {
        double px = __dmul_rn(eta, __fma_rn(cos_t, nx, udx)), py = __dmul_rn(eta, __fma_rn(cos_t, ny, udy)),
               pz = __dmul_rn(eta, __fma_rn(cos_t, nz, udz));
        double k = -__dsqrt_rn(fabs(__dsub_rn(1.0, ddot3(px, py, pz, px, py, pz))));
        dx = __fma_rn(k, nx, px);
        dy = __fma_rn(k, ny, py);
        dz = __fma_rn(k, nz, pz);
    }
    ar = ag = ab = 1.0;
    return true;
}

// sky, rrt.cu:68-75, times the path throughput
__device__ __forceinline__ void sky_d(const RayD &r, double tr, double tg, double tb, double &cr, double &cg, double &cb)
{
    double uy = __dmul_rn(r.dy, __ddiv_rn(1.0, __dsqrt_rn(ddot3(r.dx, r.dy, r.dz, r.dx, r.dy, r.dz))));
    double t = __dmul_rn(0.5, __dadd_rn(uy, 1.0));
    double w = __dsub_rn(1.0, t);
    cr = __dmul_rn(tr, __fma_rn(t, 0.5, w));
    cg = __dmul_rn(tg, __fma_rn(t, 0.7, w));
    cb = __dmul_rn(tb, __fma_rn(t, 1.0, w));
}

__device__ __forceinline__ unsigned long long to_fixed_d(double x)
{
    if (!(x > 0.0)) return 0ull;
    x = fmin(x, 1048576.0);
    return __double2ull_rn(__dmul_rn(x, 1099511627776.0));
}

} // namespace rrtb
