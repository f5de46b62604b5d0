// rrtb_device.cuh -- device-side math of the B200 path-tracing core (sm_100a).
//
// Everything a ray needs between "generate" and "accumulate": counter-based RNG, primary-ray
// generation, slab / sphere / moving-sphere / triangle tests, hit record, material scatter.
// Replaces (file:line under /root/reference):
//   curand XORWOW + wrappers        rrt.cu:81-89, rtweekend.h:80-91   -> Philox4x32-10, stateless
//   camera::get_ray                 camera.h:31-38, rrt.cu:112-114
//   aabb::hit                       aabb.h:18-93                      -> FFMA2 + FMNMX3 on 4 boxes, no divides
//   sphere::hit / moving_sphere::hit sphere.h:33-58, moving_sphere.h:27-58
//   triangle::hit                   triangle.h:35-75
//   hit_record::set_face_normal     hittable.h:16-20
//   lambertian/metal/dielectric::scatter material.h:21-32,48-57,76-109 -> type switch, no vtable
//   reflect / refract               vec3.h:156-164
//
// Rounding discipline: functions whose results are compared BIT-EXACTLY with the CPU oracle
// (oracle/rrt_oracle.c) are written with explicit round-to-nearest intrinsics (__fmaf_rn, __fmul_rn,
// __fadd_rn, __dmul_rn, __fma_rn ...) which nvcc never contracts or reassociates.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rrtb {

// -DRRTB_DEBUG_CHECKS builds librrtb200_dbg.so: invariants of the traversal stack and of the pool stacks are
// counted into a device word that rrtb_render hands back in stats.reserved (compute-sanitizer is closed on
// this GPU pool, so the bounds are checked by the code itself; tests/test_gpu_edge_cases.py).
#ifdef RRTB_DEBUG_CHECKS
__device__ unsigned int g_rrtb_violations;
#define RRTB_CHECK(cond)                              \
    do {                                              \
        if (!(cond)) atomicAdd(&g_rrtb_violations, 1u); \
    } while (0)
#else
#define RRTB_CHECK(cond) ((void)0)
#endif

// ---- scene as the kernels see it -----------------------------------------------------------------
// Leaf record: 3 x float4 (48 B) per primitive, in LEAF ORDER (Morton order for the LBVH, object-id
// order for the flat scan):
//   sphere         a = (c.xyz, r)    b = (double c.x, double c.y)  c = (double c.z, double r)   (the same values, converted once)
//   moving sphere  a = (c0.xyz, r)   b = (c1-c0 .xyz, t0)   c = (t1-t0, -, -, -)
//   triangle       a = (v0.xyz, n.x) b = (e1.xyz, n.y)      c = (e2.xyz, n.z)    n = unit face normal
//   moving tri.    a = (base.xyz, rate.x) b = (e1 base.xyz, rate.y) c = (e2 base.xyz, rate.z)   v0(time) = fma(rate, time, base)
//                  + two more float4 in the EXT array (2 per leaf slot, allocated only for scenes with moving triangles):
//                  x0 = (e1 rate.xyz, -), x1 = (e2 rate.xyz, -);  e(time) = fma(rate, time, base), a zero rate keeps its base
//                  (SURVEY 8f4, include/rrtb.h "rrtb_mtriangle"; the normal is that of the pose at the ray's time)
// leaf_info[k] = (object id, material index)
// Traversal node: a 4-WIDE node collapsed from the canonical binary LBVH (rrtb_bvh.cu k_collapse4), 24 words (96 B,
// read with three 256-bit loads): the padded boxes of the four children as centre c (float) and half extent h (fp16,
// rounded UP: the box only grows, by < 0.1 % of its half extent; +inf above 65504) and the four child refs:
//   words  0-11  c.x[0..3]  c.y[0..3]  c.z[0..3]
//   words 12-17  h.x(0,1) h.x(2,3) h.y(0,1) h.y(2,3) h.z(0,1) h.z(2,3): two fp16 per word, child 2k in the low half --
//                two HADD2.F32 (fma pipe) turn a word into the FP32x2 pair that FFMA2 takes
//   words 18-21  bits(child ref[0..3])      words 22-23 unused
// The render kernels are bound by the l1tex data stage (ncu: 81-87 % of its peak), which spends a cycle per load
// instruction and 128-byte line touched: the 128-byte all-float node of the first version cost four of them per lane
// and visit, this one three.
// child ref >= 0: wide node index;  < 0: leaf, ~ref = (leaf slot << 2) | type.  An unused child slot has
// h = -inf (its slab test can never pass) and ref = TRAV_DONE.
//
// Motion node (scenes with moving primitives and an open shutter; SURVEY 8f4): 40 words (160 B, five 256-bit loads):
// the child boxes at BOTH ends of the shutter; the traversal interpolates box(s) = (1 - s) box0 + s box1 with
// s = (ray time - shutter open) / (shutter close - open).  Primitives move linearly in time, so the interpolated
// box bounds them at every time of the shutter and is as tight as the motion allows, where a box spanning the whole
// shutter (the reference's moving_sphere::bounding_box, moving_sphere.h:60-66) grows with the distance travelled.
//   words  0-11  c0.x[4] c0.y[4] c0.z[4]        words 12-23  c1.x[4] c1.y[4] c1.z[4]
//   words 24-29  h0 pairs (as above)             words 30-35  h1 pairs        words 36-39  bits(child ref[0..3])
enum : int { PRIM_SPHERE = 0, PRIM_MSPHERE = 1, PRIM_TRIANGLE = 2, PRIM_MTRIANGLE = 3 };

struct DeviceScene {
    const float4 *wnodes;    // [6 * n_wide] 4-wide traversal nodes (96 B each), root = 0; motion: [10 * n_wide] (160 B)
    int motion;              // != 0: wnodes holds motion nodes
    float shutter_open, shutter_inv; // s = (time - shutter_open) * shutter_inv
    const float4 *leaves;    // [3 * n]   leaf order
    const int2 *leaf_info;   // [n]
    const float4 *flat_leaves; // [3 * n]  object-id order (scan mode)
    const int2 *flat_info;   // [n]
    const float4 *leaf_ext;  // [2 * n] edge rates of moving triangles, leaf order (nullptr without moving triangles)
    const float4 *flat_ext;  // [2 * n] the same in object-id order
    const float4 *materials; // [nm] (albedo.xyz, param)
    const int *material_type;// [nm]
    int n_prims, n_spheres, n_mspheres, n_triangles, n_mtriangles;
    int use_bvh;
};

struct DeviceCamera { // rrtb_camera, by value in kernel params (constant bank)
    float origin[3], llc[3], horizontal[3], vertical[3], u[3], v[3], w[3];
    float lens_radius, time0, time1;
    float inv_w1, inv_h1; // 1 / (W - 1), 1 / (H - 1)
};

struct LeafAux { // what travels with a leaf-record array: (object id, material) per slot, edge rates of moving triangles
    const int2 *info;
    const float4 *ext;
};

struct Ray {
    float ox, oy, oz, dx, dy, dz, tm;
};

struct TravCounters { // per-lane work counters of the counting build (SURVEY 8d: V_box, V_sph, V_msph, V_tri)
    unsigned long long box, sph, msph, tri;
};

struct Hit {
    float t;
    int ref; // encoded leaf ref ((slot << 2) | type), -1 = miss
    int obj; // object id (valid only after a tie was resolved or after finish)
};

// ---- Philox4x32-10 -----------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ float u01(uint32_t x) { return __fmul_rn((float)(x >> 8), 5.9604644775390625e-08f); }

// (cos, sin)(2*pi*(u - 1/2)): exact quadrant reduction + fixed FMA polynomials (bit-exact vs oracle)
__device__ __forceinline__ void sincos2pi(float u, float &co, float &si)
{
    float x = __fadd_rn(u, -0.5f);
    float qf = rintf(__fmul_rn(x, 4.0f));
    float r = __fmaf_rn(qf, -0.25f, x);
    float a = __fmul_rn(r, 6.283185307179586f);
    float a2 = __fmul_rn(a, a);
    float sp = __fmaf_rn(a2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = __fmaf_rn(a2, sp, -1.6666654611e-1f);
    float sn = __fmaf_rn(__fmul_rn(a, a2), sp, a);
    float cp = __fmaf_rn(a2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = __fmaf_rn(a2, cp, 4.166664568298827e-2f);
    cp = __fmaf_rn(a2, cp, -0.5f);
    float cs = __fmaf_rn(a2, cp, 1.0f);
    int q = (int)qf & 3;
    co = (q & 1) ? sn : cs;
    si = (q & 1) ? cs : sn;
    if (q == 1 || q == 2) co = -co;
    if (q >= 2) si = -si;
}

// ---- primary rays: rrt.cu:112-114 + camera.h:31-38 ------------------------------------------------------
__device__ __forceinline__ Ray camera_ray(const DeviceCamera &cam, int W, int H, int i, int j, int sample, uint2 key)
{
    const int pixel = j * W + i;
    uint4 b0 = philox4x32_10(make_uint4((uint32_t)pixel, (uint32_t)sample, 0u, 0u), key);
    // u = (i + xi) / (W - 1) (rrt.cu:112) as a multiplication by the host-computed reciprocal
    float u = __fmul_rn(__fadd_rn((float)i, u01(b0.x)), cam.inv_w1);
    float v = __fmul_rn(__fadd_rn((float)j, u01(b0.y)), cam.inv_h1);
    float ofx = 0.f, ofy = 0.f, ofz = 0.f;
    if (cam.lens_radius > 0.0f) {
        float r = __fmul_rn(__fsqrt_rn(u01(b0.z)), cam.lens_radius);
        float c, s;
        sincos2pi(u01(b0.w), c, s);
        float rdx = __fmul_rn(r, c), rdy = __fmul_rn(r, s);
        ofx = __fmaf_rn(cam.v[0], rdy, __fmul_rn(cam.u[0], rdx));
        ofy = __fmaf_rn(cam.v[1], rdy, __fmul_rn(cam.u[1], rdx));
        ofz = __fmaf_rn(cam.v[2], rdy, __fmul_rn(cam.u[2], rdx));
    }
    Ray r;
    r.ox = __fadd_rn(cam.origin[0], ofx);
    r.oy = __fadd_rn(cam.origin[1], ofy);
    r.oz = __fadd_rn(cam.origin[2], ofz);
    r.dx = __fsub_rn(__fsub_rn(__fmaf_rn(v, cam.vertical[0], __fmaf_rn(u, cam.horizontal[0], cam.llc[0])), cam.origin[0]), ofx);
    r.dy = __fsub_rn(__fsub_rn(__fmaf_rn(v, cam.vertical[1], __fmaf_rn(u, cam.horizontal[1], cam.llc[1])), cam.origin[1]), ofy);
    r.dz = __fsub_rn(__fsub_rn(__fmaf_rn(v, cam.vertical[2], __fmaf_rn(u, cam.horizontal[2], cam.llc[2])), cam.origin[2]), ofz);
    r.tm = cam.time0;
    if (cam.time0 != cam.time1) {
        uint4 b1 = philox4x32_10(make_uint4((uint32_t)pixel, (uint32_t)sample, 1u, 0u), key);
        r.tm = __fmaf_rn(__fsub_rn(cam.time1, cam.time0), u01(b1.x), cam.time0);
    }
    return r;
}

// ---- per-ray precomputation ------------------------------------------------------------------------------
// The slab test only has to be CONSERVATIVE (boxes are padded by 2^-20 * scene magnitude at flatten time,
// which covers the rounding of the FMA form and of the approximate reciprocal), so 1/d is one MUFU.RCP.
// Exactness lives in the leaf tests.
struct RayPre {
    float ix, iy, iz;    // ~1/d
    float oox, ooy, ooz; // -o/d
    float s;             // motion nodes only: where the ray's time lies in the shutter interval, 0 .. 1
};

__device__ __forceinline__ float rcp_approx(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ RayPre ray_pre(const Ray &r)
{
    RayPre p;
    // a direction component of (almost) exactly zero would make the FMA-form slab test compute inf - inf
    p.ix = rcp_approx(fabsf(r.dx) < 1e-20f ? copysignf(1e-20f, r.dx) : r.dx);
    p.iy = rcp_approx(fabsf(r.dy) < 1e-20f ? copysignf(1e-20f, r.dy) : r.dy);
    p.iz = rcp_approx(fabsf(r.dz) < 1e-20f ? copysignf(1e-20f, r.dz) : r.dz);
    p.oox = -r.ox * p.ix;
    p.ooy = -r.oy * p.iy;
    p.ooz = -r.oz * p.iz;
    p.s = 0.f;
    return p;
}

// sm_100a 3-input min/max (PTX ISA 8.6, SASS FMNMX3): a slab test needs 10 alu-pipe ops instead of 12
__device__ __forceinline__ float fmax3(float a, float b, float c)
{
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float fmin3(float a, float b, float c)
{
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// Packed FP32x2 arithmetic (PTX ISA 8.6 fma.rn.f32x2, SASS FFMA2): one instruction, two lanes of a 64-bit register
// pair; a pair built from one scalar twice costs nothing (ptxas encodes it as a broadcast operand `R.F32`, with
// |.| and negation as operand modifiers).
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// two fp16 in one word -> the FP32x2 pair (low half first): two HADD2.F32 (one per half, operand swizzle .H0_H0 / .H1_H1),
// which run on the fma pipe -- the bf16 pairs of the first 96-byte node cost a shift and a LOP3 per word on the alu pipe,
// the pipe that bounds a node visit (profiles/README.md)
__device__ __forceinline__ f32x2 half2x2(float word)
{
    float lo, hi;
    asm("{\n\t.reg .b16 a, b;\n\tmov.b32 {a, b}, %2;\n\tcvt.f32.f16 %0, a;\n\tcvt.f32.f16 %1, b;\n\t}"
        : "=f"(lo), "=f"(hi)
        : "r"(__float_as_uint(word)));
    return pack2(lo, hi);
}

// Slab test of TWO children of a wide node at once (already padded boxes as centre c and half extent h; each
// f32x2 holds the same component of the two children); inclusive; entry distances in ta / tb.  Per axis
// t_c = (c - o)/d, [t_c - h|1/d|, t_c + h|1/d|]: three FFMA2 for the two boxes (no min/max to order the planes;
// ptxas folds the negation and the |.| of the broadcast scalar into operand modifiers), then per box
// 2 FMNMX3 + 2 FMNMX + 1 FSETP.  The scalar form cost 24 fma-pipe + 10 alu-pipe instructions per pair, the
// min/max form before it 12 + 22 on the alu pipe that ncu showed as the busiest unit.
__device__ __forceinline__ void box_hit_pair(f32x2 cx, f32x2 cy, f32x2 cz, f32x2 hx, f32x2 hy, f32x2 hz, const RayPre &p,
                                             float t_min, float t_max, bool &ha, bool &hb, float &ta, float &tb)
{
    const float ax = fabsf(p.ix), ay = fabsf(p.iy), az = fabsf(p.iz);
    const f32x2 tx = fma2(cx, pack2(p.ix, p.ix), pack2(p.oox, p.oox));
    const f32x2 ty = fma2(cy, pack2(p.iy, p.iy), pack2(p.ooy, p.ooy));
    const f32x2 tz = fma2(cz, pack2(p.iz, p.iz), pack2(p.ooz, p.ooz));
    const f32x2 ux = mul2(hx, pack2(ax, ax));
    const f32x2 uy = mul2(hy, pack2(ay, ay));
    const f32x2 uz = mul2(hz, pack2(az, az));
    float lxa, lxb, lya, lyb, lza, lzb, hxa, hxb, hya, hyb, hza, hzb;
    unpack2(sub2(tx, ux), lxa, lxb);
    unpack2(sub2(ty, uy), lya, lyb);
    unpack2(sub2(tz, uz), lza, lzb);
    unpack2(add2(tx, ux), hxa, hxb);
    unpack2(add2(ty, uy), hya, hyb);
    unpack2(add2(tz, uz), hza, hzb);
    ta = fmaxf(fmax3(lxa, lya, lza), t_min);
    tb = fmaxf(fmax3(lxb, lyb, lzb), t_min);
    ha = ta <= fminf(fmin3(hxa, hya, hza), t_max);
    hb = tb <= fminf(fmin3(hxb, hyb, hzb), t_max);
}

// ---- primitive tests (bit-exact vs oracle sphere_roots / triangle_t) ---------------------------------------
// sphere.h:33-58: nearest root in [t_min, t_max], inclusive.  oc, half_b, c and the discriminant in
// double (the cancellation-prone part), roots in float via the cancellation-free pair q/a, c/q.
// (cx, cy, cz, rr): centre and radius in double -- exact conversions of the float scene values, which static spheres carry
// in the 32 spare bytes of their leaf record so that the test converts only the ray (6 instead of 10 F2F on the XU pipe,
// the pipe that bounds a sphere test: 17 XU instructions of 8 cycles each in ~75)
__device__ __forceinline__ bool sphere_test_d4(const Ray &r, double cx, double cy, double cz, double rr, float t_min,
                                               float t_max, float &t_out)
{
    double ocx = __dsub_rn((double)r.ox, cx);
    double ocy = __dsub_rn((double)r.oy, cy);
    double ocz = __dsub_rn((double)r.oz, cz);
    double dx = r.dx, dy = r.dy, dz = r.dz;
    double a = __fma_rn(dz, dz, __fma_rn(dy, dy, __dmul_rn(dx, dx)));
    double hb = __fma_rn(ocz, dz, __fma_rn(ocy, dy, __dmul_rn(ocx, dx)));
    double cc = __fma_rn(-rr, rr, __fma_rn(ocz, ocz, __fma_rn(ocy, ocy, __dmul_rn(ocx, ocx))));
    double disc = __fma_rn(-a, cc, __dmul_rn(hb, hb));
    if (disc < 0.0) return false;
    float sq = __fsqrt_rn(__double2float_rn(disc));
    float hbf = __double2float_rn(hb), ccf = __double2float_rn(cc);
    float q = -__fadd_rn(hbf, copysignf(sq, hbf));
    float r0 = __fdiv_rn(q, __double2float_rn(a)), r1 = __fdiv_rn(ccf, q);
    float tn = fminf(r0, r1), tf = fmaxf(r0, r1);
    float root = tn;
    if (!(root >= t_min && root <= t_max)) {
        root = tf;
        if (!(root >= t_min && root <= t_max)) return false;
    }
    t_out = root;
    return true;
}
__device__ __forceinline__ bool sphere_test(const Ray &r, const RayPre &, float cx, float cy, float cz, float rad,
                                            float t_min, float t_max, float &t_out)
{
    return sphere_test_d4(r, (double)cx, (double)cy, (double)cz, (double)rad, t_min, t_max, t_out);
}

// moving_sphere.h:27-30
__device__ __forceinline__ void msphere_center(float4 a, float4 b, float4 c, float time, float &cx, float &cy, float &cz)
{
    float k = __fdiv_rn(__fsub_rn(time, b.w), c.x);
    cx = __fmaf_rn(k, b.x, a.x);
    cy = __fmaf_rn(k, b.y, a.y);
    cz = __fmaf_rn(k, b.z, a.z);
}

__device__ __forceinline__ double dcross(double a, double b, double c, double d)
{
    return __fma_rn(a, b, -__dmul_rn(c, d));
}

__device__ __forceinline__ float dot3_rn(float ax, float ay, float az, float bx, float by, float bz)
{
    return __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
}
__device__ __forceinline__ void unit3_rn(float &x, float &y, float &z)
{
    float inv = __fdiv_rn(1.0f, __fsqrt_rn(dot3_rn(x, y, z, x, y, z)));
    x = __fmul_rn(inv, x);
    y = __fmul_rn(inv, y);
    z = __fmul_rn(inv, z);
}
// triangle.h:9-15: unit(cross(unit(v1-v0), unit(v2-v0)))
__device__ __forceinline__ void triangle_unit_normal(float ax, float ay, float az, float bx, float by, float bz, float &nx,
                                                     float &ny, float &nz)
{
    unit3_rn(ax, ay, az);
    unit3_rn(bx, by, bz);
    nx = __fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by));
    ny = __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz));
    nz = __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx));
    unit3_rn(nx, ny, nz);
}

// out of line: only moving triangles recompute their normal at shading time, and the three normalisations would
// otherwise sit in the middle of every kernel's shading code
static __device__ __noinline__ float3 triangle_unit_normal_cold(float4 b, float4 c)
{
    float3 n;
    triangle_unit_normal(b.x, b.y, b.z, c.x, c.y, c.z, n.x, n.y, n.z);
    return n;
}

// edges of a moving triangle's pose at `time` (include/rrtb.h "rrtb_mtriangle"): e(t) = fma(rate, t, base) in float, a
// zero rate keeps its base exactly (so a translating instance has bit for bit the edges of the static one)
__device__ __forceinline__ float lin_at(float rate, float time, float base)
{
    return rate == 0.0f ? base : __fmaf_rn(rate, time, base);
}
__device__ __forceinline__ void mtri_edges(const float4 *__restrict__ ext, int slot, float time, float4 &b, float4 &c)
{
    const float4 x0 = __ldg(ext + 2 * (size_t)(unsigned)slot), x1 = __ldg(ext + 2 * (size_t)(unsigned)slot + 1);
    b.x = lin_at(x0.x, time, b.x);
    b.y = lin_at(x0.y, time, b.y);
    b.z = lin_at(x0.z, time, b.z);
    c.x = lin_at(x1.x, time, c.x);
    c.y = lin_at(x1.y, time, c.y);
    c.z = lin_at(x1.z, time, c.z);
}

// triangle.h:35-75: Moeller-Trumbore, numerators in double, division-free barycentric tests, exclusive range.
// (v0x, v0y, v0z) is the first vertex in double: the stored one, or v0(time) of a translating instance triangle.
__device__ __forceinline__ bool triangle_test(const Ray &r, double v0x, double v0y, double v0z, float4 B, float4 C,
                                              float t_min, float t_max, float &t_out)
{
    const double EPS = (double)1e-7f;
    double e1x = B.x, e1y = B.y, e1z = B.z, e2x = C.x, e2y = C.y, e2z = C.z;
    double dx = r.dx, dy = r.dy, dz = r.dz;
    double hx = dcross(dy, e2z, dz, e2y), hy = dcross(dz, e2x, dx, e2z), hz = dcross(dx, e2y, dy, e2x);
    double det = __fma_rn(e1z, hz, __fma_rn(e1y, hy, __dmul_rn(e1x, hx)));
    if (det > -EPS && det < EPS) return false;
    double sx = __dsub_rn((double)r.ox, v0x), sy = __dsub_rn((double)r.oy, v0y), sz = __dsub_rn((double)r.oz, v0z);
    double un = __fma_rn(sz, hz, __fma_rn(sy, hy, __dmul_rn(sx, hx)));
    double qx = dcross(sy, e1z, sz, e1y), qy = dcross(sz, e1x, sx, e1z), qz = dcross(sx, e1y, sy, e1x);
    double vn = __fma_rn(dz, qz, __fma_rn(dy, qy, __dmul_rn(dx, qx)));
    if (det > 0.0) {
        if (un < 0.0 || un > det || vn < 0.0 || __dadd_rn(un, vn) > det) return false;
    }
    else {
        if (un > 0.0 || un < det || vn > 0.0 || __dadd_rn(un, vn) < det) return false;
    }
    double tn = __fma_rn(e2z, qz, __fma_rn(e2y, qy, __dmul_rn(e2x, qx)));
    float t = __fdiv_rn(__double2float_rn(tn), __double2float_rn(det));
    // triangle.h:61 is exclusive at both ends; an exact tie with the current closest hit (t == t_max) is let
    // through and settled by candidate_wins, which restates that exclusivity order-independently
    if (t > 1e-7f && t > t_min && t <= t_max) {
        t_out = t;
        return true;
    }
    return false;
}

// Order-independent form of the flat scan's tie rule (hittable_list.h:102-114 with the inclusive sphere
// range and exclusive triangle range): at exactly equal t the LAST sphere-like object in id order wins,
// else the FIRST triangle.
__device__ __forceinline__ bool candidate_wins(float t, int type, int obj, float bt, int btype, int bobj)
{
    if (bobj < 0) return true;
    if (t < bt) return true;
    if (t > bt) return false;
    bool ct = type >= PRIM_TRIANGLE, bt_tri = btype >= PRIM_TRIANGLE; // moving triangles are triangles
    if (ct != bt_tri) return !ct;
    return ct ? (obj < bobj) : (obj > bobj);
}

// Test leaf `slot` (type known) and update the running closest hit.
template <bool COUNT, bool MTRI = true>
__device__ __forceinline__ void leaf_test(const float4 *__restrict__ leaves, const LeafAux info, int slot,
                                          int type, const Ray &r, const RayPre &p, float t_min, Hit &best,
                                          TravCounters &cnt)
{
    if (COUNT) {
        if (type == PRIM_SPHERE) ++cnt.sph;
        else if (type == PRIM_MSPHERE) ++cnt.msph;
        else ++cnt.tri;
    }
    const float4 *rec = leaves + (size_t)(unsigned)slot * 3u; // one IMAD.WIDE (slot * 48 + base)
    float t;
    bool h;
    if (type == PRIM_SPHERE) { // centre and radius as doubles in the second and third float4 (k_prepare)
        const float4 b = __ldg(rec + 1), c = __ldg(rec + 2);
        h = sphere_test_d4(r, __hiloint2double(__float_as_int(b.y), __float_as_int(b.x)),
                           __hiloint2double(__float_as_int(b.w), __float_as_int(b.z)),
                           __hiloint2double(__float_as_int(c.y), __float_as_int(c.x)),
                           __hiloint2double(__float_as_int(c.w), __float_as_int(c.z)), t_min, best.t, t);
    }
    else if (type == PRIM_MSPHERE) {
        float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
        float cx, cy, cz;
        msphere_center(a, b, c, r.tm, cx, cy, cz);
        h = sphere_test(r, p, cx, cy, cz, a.w, t_min, best.t, t);
    }
    else {
        float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
        double v0x = a.x, v0y = a.y, v0z = a.z;
        if (MTRI && type == PRIM_MTRIANGLE) { // the instance moves: meet the triangle of the pose at the ray's time
            double tm = r.tm;
            v0x = __fma_rn((double)a.w, tm, v0x);
            v0y = __fma_rn((double)b.w, tm, v0y);
            v0z = __fma_rn((double)c.w, tm, v0z);
            mtri_edges(info.ext, slot, r.tm, b, c);
        }
        h = triangle_test(r, v0x, v0y, v0z, b, c, t_min, best.t, t);
    }
    if (!h) return;
    if (best.ref >= 0 && t == best.t) { // exact tie: resolve by object id (rare path)
        int obj = __ldg(&info.info[slot]).x;
        int bobj = __ldg(&info.info[best.ref >> 2]).x;
        if (!candidate_wins(t, type, obj, best.t, best.ref & 3, bobj)) return;
    }
    best.t = t;
    best.ref = (slot << 2) | type;
}

// ---- closest hit: traversal of the 4-wide tree (replaces bvh_node::hit recursion, bvh.h:167-175) -----------
// Iterative and STEP-WISE so that a warp-level scheduler can interleave it with other work:
//   cur >= 0          wide node to visit      -> wide_step: one 128-byte node fetch tests four children; the
//                     nearest hit child is next, the other hit children are pushed
//   cur <  0          a leaf reference        -> leaf_step (rrtb_path.cuh): exact primitive test, then pop
//   cur == TRAV_DONE  traversal finished
// Every child that is hit gets a KEY = the bits of its entry distance with the low mantissa BYTE replaced by its slot
// (one PRMT; the 15 mantissa bits that remain order the children): non-negative floats order as integers, so the nearest
// child is one 4-input unsigned minimum (2 VIMNMX3), its slot comes with it, and equal distances can not tie.  The other
// hit children are pushed in slot order.  A visit is branch-free: pushes, selection and the pop of a visit that hit no
// child are predicated instructions (the branch around the pushes diverged in most warps and cost five instructions).
// Measured and dropped (profiles/README.md, round 2): pushing the keys with the references so that a leaf whose
// entry distance already exceeds the closest hit is skipped at pop time (-12 % leaf tests, but twice the local-memory
// traffic: 5 % slower), a full sort of the hit children (more instructions than the visits it saves), and the
// binary tree itself (two children per node: 3 % slower on the headline scene, 10 % on the 1.1 M-primitive one).
// A collapsed tree is never deeper than the binary tree it comes from: <= 62 levels for the Karras tree (30-bit
// Morton codes with an index tie-break), and the SAH rebuild of its lower subtrees (rrtb_bvh.cu k_sah_rebuild) keeps
// every leaf within 63 levels; a visit pushes at most three entries, so 192 entries (one of them the TRAV_DONE at the
// bottom) can not overflow.  The entries live in local memory (L1-resident).
#define RRTB_WIDTH 4
#define RRTB_NODE_F4 6 // float4 per traversal node (96 B)
#define RRTB_MOTION_NODE_F4 10 // float4 per motion node (160 B)
#define RRTB_STACK 192
#define TRAV_DONE ((int)0x80000000)
#define KEY_MISS (-1) // as unsigned the largest key, as signed below every real key

// 32-byte read-only load (PTX ISA 8.8 ld.global.nc.v8.f32, SASS LDG.E.256.CONSTANT; p must be 32-byte aligned)
__device__ __forceinline__ void ldg256(const float4 *p, float4 &a, float4 &b)
{
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
        : "l"(p));
}

// The stack grows upwards from stk[1]; stk[0] holds TRAV_DONE, so the pop that empties the stack ends the traversal
// without a test.  TravSp points at the next free entry (a local-memory address kept in a register instead of an index
// that every access scales and adds to the frame: 218 -> 196 SASS instructions per two visits together with the
// branch-free visit and the PRMT keys; measured with the round-1 forms as variant builds, profiles/README.md).
typedef int *TravSp;
__device__ __forceinline__ void trav_pop(int &cur, TravSp &sp, const int *) { cur = *--sp; }
__device__ __forceinline__ void trav_pop_if_neg(int m, int &cur, TravSp &sp, const int *)
{
    if (m < 0) cur = *--sp;
}
__device__ __forceinline__ void trav_push_if_gt(int k, int m, TravSp &sp, int *, int ref)
{
    if (k > m) *sp++ = ref;
}
// start a traversal at the root
__device__ __forceinline__ void trav_begin(int &cur, TravSp &sp, int *stk)
{
    cur = 0;
    stk[0] = TRAV_DONE;
    sp = stk + 1;
}
__device__ __forceinline__ int trav_depth(TravSp sp, const int *stk) { return (int)(sp - stk); }

// t_min must be >= 0 (keys order as integers only for non-negative distances); rrtb_trace_closest checks it
// (1 - s) a + s b on an FP32x2 pair
__device__ __forceinline__ f32x2 lerp2(f32x2 a, f32x2 b, float s, float oms)
{
    return fma2(b, pack2(s, s), mul2(a, pack2(oms, oms)));
}

template <bool COUNT, bool MOTION = false>
__device__ __forceinline__ void wide_step(const float4 *__restrict__ wnodes, const RayPre &p, float t_min, float t_max,
                                          int &cur, TravSp &sp, int *stk, TravCounters &cnt)
{
    if (COUNT) cnt.box += RRTB_WIDTH;
    bool h0, h1, h2, h3;
    float t0, t1, t2, t3;
    int4 rf;
    if (MOTION) {
        const float4 *q = wnodes + (size_t)(unsigned)cur * (unsigned)RRTB_MOTION_NODE_F4;
        float4 ax, ay, az, bx, by, bz, g0, g1, g2, rr;
        ldg256(q, ax, ay);     // c0.x[4] c0.y[4]
        ldg256(q + 2, az, bx); // c0.z[4] c1.x[4]
        ldg256(q + 4, by, bz); // c1.y[4] c1.z[4]
        ldg256(q + 6, g0, g1); // fp16 pairs h0.x(0,1) h0.x(2,3) h0.y(0,1) h0.y(2,3) | h0.z(0,1) h0.z(2,3) h1.x(0,1) h1.x(2,3)
        ldg256(q + 8, g2, rr); // fp16 pairs h1.y(0,1) h1.y(2,3) h1.z(0,1) h1.z(2,3) | refs
        rf = make_int4(__float_as_int(rr.x), __float_as_int(rr.y), __float_as_int(rr.z), __float_as_int(rr.w));
        const float s = p.s, oms = 1.0f - p.s;
        box_hit_pair(lerp2(pack2(ax.x, ax.y), pack2(bx.x, bx.y), s, oms), lerp2(pack2(ay.x, ay.y), pack2(by.x, by.y), s, oms),
                     lerp2(pack2(az.x, az.y), pack2(bz.x, bz.y), s, oms), lerp2(half2x2(g0.x), half2x2(g1.z), s, oms),
                     lerp2(half2x2(g0.z), half2x2(g2.x), s, oms), lerp2(half2x2(g1.x), half2x2(g2.z), s, oms), p, t_min, t_max, h0, h1, t0, t1);
        box_hit_pair(lerp2(pack2(ax.z, ax.w), pack2(bx.z, bx.w), s, oms), lerp2(pack2(ay.z, ay.w), pack2(by.z, by.w), s, oms),
                     lerp2(pack2(az.z, az.w), pack2(bz.z, bz.w), s, oms), lerp2(half2x2(g0.y), half2x2(g1.w), s, oms),
                     lerp2(half2x2(g0.w), half2x2(g2.y), s, oms), lerp2(half2x2(g1.y), half2x2(g2.w), s, oms), p, t_min, t_max, h2, h3, t2, t3);
    }
    else {
        // the index is widened before it is scaled so that the address is ONE IMAD.WIDE (cur * 96 + base)
        const float4 *q = wnodes + (size_t)(unsigned)cur * (unsigned)RRTB_NODE_F4;
        float4 cx, cy, cz, hw, zr, rs;
        ldg256(q, cx, cy);     // c.x[4] c.y[4]
        ldg256(q + 2, cz, hw); // c.z[4], fp16 pairs h.x(0,1) h.x(2,3) h.y(0,1) h.y(2,3)
        ldg256(q + 4, zr, rs); // fp16 pairs h.z(0,1) h.z(2,3), ref[0..1] | ref[2..3], unused
        rf = make_int4(__float_as_int(zr.z), __float_as_int(zr.w), __float_as_int(rs.x), __float_as_int(rs.y));
        box_hit_pair(pack2(cx.x, cx.y), pack2(cy.x, cy.y), pack2(cz.x, cz.y), half2x2(hw.x), half2x2(hw.z), half2x2(zr.x), p, t_min, t_max,
                     h0, h1, t0, t1);
        box_hit_pair(pack2(cx.z, cx.w), pack2(cy.z, cy.w), pack2(cz.z, cz.w), half2x2(hw.y), half2x2(hw.w), half2x2(zr.y), p, t_min, t_max,
                     h2, h3, t2, t3);
    }
    // the slot replaces the low BYTE of the distance (one PRMT per child; 15 mantissa bits order the children)
    const int k0 = h0 ? (int)__byte_perm(__float_as_uint(t0), 0x03020100u, 0x3214u) : KEY_MISS;
    const int k1 = h1 ? (int)__byte_perm(__float_as_uint(t1), 0x03020100u, 0x3215u) : KEY_MISS;
    const int k2 = h2 ? (int)__byte_perm(__float_as_uint(t2), 0x03020100u, 0x3216u) : KEY_MISS;
    const int k3 = h3 ? (int)__byte_perm(__float_as_uint(t3), 0x03020100u, 0x3217u) : KEY_MISS;
    // unsigned minimum: a real key (non-negative float bits) beats KEY_MISS
    const int m = (int)min(min((unsigned)k0, (unsigned)k1), min((unsigned)k2, (unsigned)k3));
    // SIGNED k > m: false for the nearest (equal) and for a miss (-1)
    RRTB_CHECK(trav_depth(sp, stk) >= 0 && trav_depth(sp, stk) + 3 <= RRTB_STACK);
    trav_push_if_gt(k0, m, sp, stk, rf.x);
    trav_push_if_gt(k1, m, sp, stk, rf.y);
    trav_push_if_gt(k2, m, sp, stk, rf.z);
    trav_push_if_gt(k3, m, sp, stk, rf.w);
    cur = rf.w;
    if (k2 == m) cur = rf.z;
    if (k1 == m) cur = rf.y;
    if (k0 == m) cur = rf.x;
    // no child hit (every key is KEY_MISS: nothing was pushed above): pop, as predicated instructions instead of a
    // divergent branch around the pushes
    trav_pop_if_neg(m, cur, sp, stk);
}

// ---- hit record: sphere.h:51-55, moving_sphere.h:51-55, triangle.h:62-66, hittable.h:16-20 ----------------
struct HitRecord {
    float px, py, pz, nx, ny, nz;
    bool front;
    int obj, mat;
};

// MTRI = false compiles the moving-triangle cases out (the pool kernel picks the variant per scene: the dead
// branches alone cost 1 % on the headline workload)
template <bool MTRI = true>
__device__ __forceinline__ HitRecord hit_record(const float4 *__restrict__ leaves, const LeafAux info,
                                                const Ray &r, const Hit &h)
{
    HitRecord rec;
    int slot = h.ref >> 2, type = h.ref & 3;
    rec.px = __fmaf_rn(h.t, r.dx, r.ox);
    rec.py = __fmaf_rn(h.t, r.dy, r.oy);
    rec.pz = __fmaf_rn(h.t, r.dz, r.oz);
    float4 a = __ldg(leaves + 3 * slot);
    if (type == PRIM_TRIANGLE) {
        float4 b = __ldg(leaves + 3 * slot + 1), c = __ldg(leaves + 3 * slot + 2);
        rec.nx = a.w;
        rec.ny = b.w;
        rec.nz = c.w;
    }
    else if (MTRI && type == PRIM_MTRIANGLE) { // the face normal of the pose at the ray's time
        float4 b = __ldg(leaves + 3 * slot + 1), c = __ldg(leaves + 3 * slot + 2);
        mtri_edges(info.ext, slot, r.tm, b, c);
        float3 n = triangle_unit_normal_cold(b, c);
        rec.nx = n.x;
        rec.ny = n.y;
        rec.nz = n.z;
    }
    else {
        float cx = a.x, cy = a.y, cz = a.z;
        if (type == PRIM_MSPHERE) {
            float4 b = __ldg(leaves + 3 * slot + 1), c = __ldg(leaves + 3 * slot + 2);
            msphere_center(a, b, c, r.tm, cx, cy, cz);
        }
        float inv = __frcp_rn(a.w);
        rec.nx = __fmul_rn(inv, __fsub_rn(rec.px, cx));
        rec.ny = __fmul_rn(inv, __fsub_rn(rec.py, cy));
        rec.nz = __fmul_rn(inv, __fsub_rn(rec.pz, cz));
    }
    float dn = __fadd_rn(__fadd_rn(__fmul_rn(r.dx, rec.nx), __fmul_rn(r.dy, rec.ny)), __fmul_rn(r.dz, rec.nz));
    rec.front = dn < 0.0f;
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

// ---- materials ------------------------------------------------------------------------------------------
// One Philox block per bounce (see oracle/rrt_oracle.c "materials" for the stream layout).  The scatter
// code may use fast reciprocal-sqrt: its results are compared with the oracle to a tolerance, not bitwise.
__device__ __forceinline__ void sample_unit_sphere(float x0, float x1, float &ux, float &uy, float &uz)
{
    float z = fmaf(-2.0f, x0, 1.0f);
    float rr = sqrtf(fmaxf(0.0f, fmaf(-z, z, 1.0f)));
    float c, s;
    sincos2pi(x1, c, s);
    ux = rr * c;
    uy = rr * s;
    uz = z;
}

// returns true if the path continues; (dx,dy,dz) = scattered direction, (ar,ag,ab) = attenuation
__device__ __forceinline__ bool scatter(int mtype, float4 m, const Ray &r, const HitRecord &rec, uint4 rnd, float &dx,
                                        float &dy, float &dz, float &ar, float &ag, float &ab)
{
    const float nx = rec.nx, ny = rec.ny, nz = rec.nz;
    if (mtype == 0) { // lambertian, material.h:21-32
        float ux, uy, uz;
        sample_unit_sphere(u01(rnd.x), u01(rnd.y), ux, uy, uz);
        dx = nx + ux;
        dy = ny + uy;
        dz = nz + uz;
        if (fabsf(dx) < 1e-8f && fabsf(dy) < 1e-8f && fabsf(dz) < 1e-8f) {
            dx = nx;
            dy = ny;
            dz = nz;
        }
        ar = m.x;
        ag = m.y;
        ab = m.z;
        return true;
    }
    float inv = rsqrtf(fmaf(r.dz, r.dz, fmaf(r.dy, r.dy, r.dx * r.dx)));
    float udx = r.dx * inv, udy = r.dy * inv, udz = r.dz * inv;
    float dn = fmaf(udz, nz, fmaf(udy, ny, udx * nx));
    if (mtype == 1) { // metal, material.h:48-57
        float k = -2.0f * dn;
        dx = fmaf(k, nx, udx);
        dy = fmaf(k, ny, udy);
        dz = fmaf(k, nz, udz);
        float fuzz = fminf(m.w, 1.0f);
        if (fuzz > 0.0f) {
            float ux, uy, uz;
            sample_unit_sphere(u01(rnd.x), u01(rnd.y), ux, uy, uz);
            float ra = u01(rnd.z);
            float rb = (float)(rnd.w >> 16) * 1.52587890625e-05f;
            float rc = (float)(rnd.w & 0xFFFFu) * 1.52587890625e-05f;
            float rad = fmaxf(ra, fmaxf(rb, rc)) * fuzz;
            dx = fmaf(rad, ux, dx);
            dy = fmaf(rad, uy, dy);
            dz = fmaf(rad, uz, dz);
        }
        ar = m.x;
        ag = m.y;
        ab = m.z;
        return fmaf(dz, nz, fmaf(dy, ny, dx * nx)) > 0.0f;
    }
    // dielectric, material.h:76-109 + vec3.h:158-164
    float ir = m.w;
    float eta = rec.front ? __frcp_rn(ir) : ir;
    float cos_t = fminf(-dn, 1.0f);
    float sin_t = sqrtf(fmaxf(0.0f, fmaf(-cos_t, cos_t, 1.0f)));
    bool cannot = eta * sin_t > 1.0f;
    float r0 = __fdividef(1.0f - eta, 1.0f + eta);
    r0 = r0 * r0;
    float om = 1.0f - cos_t;
    float om2 = om * om;
    float refl_p = fmaf(1.0f - r0, om2 * om2 * om, r0);
    if (cannot || refl_p > u01(rnd.x)) {
        float k = -2.0f * dn;
        dx = fmaf(k, nx, udx);
        dy = fmaf(k, ny, udy);
        dz = fmaf(k, nz, udz);
    }
    else {
        float px = eta * fmaf(cos_t, nx, udx), py = eta * fmaf(cos_t, ny, udy), pz = eta * fmaf(cos_t, nz, udz);
        float k = -sqrtf(fabsf(1.0f - fmaf(pz, pz, fmaf(py, py, px * px))));
        dx = fmaf(k, nx, px);
        dy = fmaf(k, ny, py);
        dz = fmaf(k, nz, pz);
    }
    ar = ag = ab = 1.0f;
    return true;
}

// sky, rrt.cu:68-75
__device__ __forceinline__ void sky(const Ray &r, float &cr, float &cg, float &cb)
{
    float inv = rsqrtf(fmaf(r.dz, r.dz, fmaf(r.dy, r.dy, r.dx * r.dx)));
    float t = 0.5f * fmaf(r.dy, inv, 1.0f);
    float w = 1.0f - t;
    cr = fmaf(t, 0.5f, w);
    cg = fmaf(t, 0.7f, w);
    cb = fmaf(t, 1.0f, w);
}

// radiance -> 2^40 fixed point (integer accumulation is associative => bit-reproducible images under
// any scheduling, sharding or reduction order)
__device__ __forceinline__ unsigned long long to_fixed(float x)
{
    if (!(x > 0.0f)) return 0ull;
    x = fminf(x, 1048576.0f);
    return __double2ull_rn((double)x * 1099511627776.0);
}

} // namespace rrtb
