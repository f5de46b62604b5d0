/* rrt_oracle.c -- TEST INFRASTRUCTURE ONLY (see rrt_oracle.h for the rules and the parity status).
 *
 * Plain C11, scalar, compiled with -ffp-contract=off so that every floating-point operation below
 * is exactly one IEEE-754 rounding; where the CUDA product uses a fused multiply-add the oracle
 * calls fma()/fmaf() explicitly.  Reference citations are file:line under /root/reference.
 */
#include "rrt_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------------------------------
 * Philox4x32-10  (Salmon, Moraes, Dror, Shaw: "Parallel Random Numbers: As Easy as 1, 2, 3", SC'11)
 * replaces curand XORWOW state (rrt.cu:81-89, rtweekend.h:80-91).
 * ---------------------------------------------------------------------------------------------- */
#define PHILOX_M0 0xD2511F53u
#define PHILOX_M1 0xCD9E8D57u
#define PHILOX_W0 0x9E3779B9u
#define PHILOX_W1 0xBB67AE85u

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int round = 0; round < 10; ++round) {
        uint64_t p0 = (uint64_t)PHILOX_M0 * c0;
        uint64_t p1 = (uint64_t)PHILOX_M1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n1 = lo1;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        uint32_t n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += PHILOX_W0;
        k1 += PHILOX_W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

float orc_u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; /* 2^-24 */ }

/* stream layout shared with the product (DESIGN.md "RNG"): ctr = (pixel, sample, dimension block, 0),
 * key = (seed lo, seed hi).  Block 0: jitter u, jitter v, lens r, lens phi.  Block 1: shutter time.
 * Block 2+b: bounce b. */
static void rng_block(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t dim, uint32_t out[4])
{
    uint32_t ctr[4] = {pixel, sample, dim, 0u};
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    orc_philox4x32_10(ctr, key, out);
}

/* cos/sin of phi = 2*pi*(u-0.5), u in [0,1).  Quadrant reduction is exact; the polynomials are
 * fixed fmaf chains, so CPU and GPU agree bit for bit. */
void orc_sincos2pi(float u, float *c, float *s)
{
    float x = u - 0.5f;                 /* exact, [-0.5, 0.5) */
    float qf = rintf(x * 4.0f);         /* -2..2 */
    float r = fmaf(qf, -0.25f, x);      /* exact, [-1/8, 1/8] */
    float a = r * 6.283185307179586f;   /* [-pi/4, pi/4] */
    float a2 = a * a;
    /* sin: a + a^3 (S1 + a2 (S2 + a2 S3)) ; cos: 1 + a2 (C1 + a2 (C2 + a2 (C3 + a2 C4))) */
    float sp = fmaf(a2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = fmaf(a2, sp, -1.6666654611e-1f);
    float sn = fmaf(a * a2, sp, a);
    float cp = fmaf(a2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = fmaf(a2, cp, 4.166664568298827e-2f);
    cp = fmaf(a2, cp, -0.5f);
    float cs = fmaf(a2, cp, 1.0f);
    int q = (int)qf & 3; /* two's complement: -1 -> 3, -2 -> 2 */
    float co, si;
    switch (q) {
    case 0: co = cs; si = sn; break;
    case 1: co = -sn; si = cs; break;
    case 2: co = -cs; si = -sn; break;
    default: co = sn; si = -cs; break;
    }
    *c = co;
    *s = si;
}

/* ------------------------------------------------------------------------------------------------
 * small float vector helpers (one rounding per operation)
 * ---------------------------------------------------------------------------------------------- */
typedef struct { float x, y, z; } f3;
static inline f3 F3(float x, float y, float z) { f3 r = {x, y, z}; return r; }
static inline f3 ld3(const float *p) { return F3(p[0], p[1], p[2]); }
static inline void st3(float *p, f3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
static inline f3 add3(f3 a, f3 b) { return F3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline f3 sub3(f3 a, f3 b) { return F3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline f3 scl3(float t, f3 a) { return F3(t * a.x, t * a.y, t * a.z); }
static inline float dot3(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline f3 cross3(f3 u, f3 v)
{
    return F3(u.y * v.z - u.z * v.y, u.z * v.x - u.x * v.z, u.x * v.y - u.y * v.x);
}
static inline f3 unit3(f3 v) /* vec3.h: unit_vector = (1/len) * v */
{
    float inv = 1.0f / sqrtf(dot3(v, v));
    return scl3(inv, v);
}

/* ------------------------------------------------------------------------------------------------
 * camera (camera.h:8-29): the reference's float build, including its double-precision tan()
 * ---------------------------------------------------------------------------------------------- */
void orc_camera_derive(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov,
                       float aspect, float aperture, float focus, float t0, float t1, rrtb_camera *out)
{
    const float pi_f = (float)3.1415926535897932385;     /* rtweekend.h:56 */
    float theta = vfov * pi_f / 180.0f;                  /* rtweekend.h:60 */
    float h = (float)tan((double)(theta / 2.0f));        /* camera.h:13: ::tan(double) then narrowed */
    float viewport_height = 2.0f * h;
    float viewport_width = aspect * viewport_height;
    f3 from = ld3(lookfrom), at = ld3(lookat), up = ld3(vup);
    f3 w = unit3(sub3(from, at));
    f3 u = unit3(cross3(up, w));
    f3 v = cross3(w, u);
    f3 horizontal = scl3(focus * viewport_width, u);
    f3 vertical = scl3(focus * viewport_height, v);
    /* origin - horizontal/2 - vertical/2 - focus*w ; operator/ is (1/t)*v (vec3.h) */
    f3 llc = sub3(sub3(sub3(from, scl3(1.0f / 2.0f, horizontal)), scl3(1.0f / 2.0f, vertical)), scl3(focus, w));
    st3(out->origin, from);
    st3(out->lower_left_corner, llc);
    st3(out->horizontal, horizontal);
    st3(out->vertical, vertical);
    st3(out->u, u);
    st3(out->v, v);
    st3(out->w, w);
    out->lens_radius = aperture / 2.0f;
    out->time0 = t0;
    out->time1 = t1;
}

/* rrt.cu:112-114 + camera.h:31-38.  The lens disk is sampled by (sqrt(xi3), 2*pi*xi4) instead of the
 * reference's rejection loop (vec3.h:127-134): same distribution, fixed number of random numbers. */
void orc_camera_ray(const rrtb_camera *cam, int W, int H, int pixel, int sample, uint64_t seed, float *ray7)
{
    uint32_t b0[4];
    rng_block(seed, (uint32_t)pixel, (uint32_t)sample, 0u, b0);
    int i = pixel % W, j = pixel / W;
    /* rrt.cu:112-113 divides by (W-1); both sides multiply by the correctly rounded reciprocal instead */
    float u = ((float)i + orc_u01(b0[0])) * (1.0f / (float)(W - 1));
    float v = ((float)j + orc_u01(b0[1])) * (1.0f / (float)(H - 1));
    f3 offset = F3(0.f, 0.f, 0.f);
    if (cam->lens_radius > 0.0f) {
        float r = sqrtf(orc_u01(b0[2])) * cam->lens_radius;
        float c, s;
        orc_sincos2pi(orc_u01(b0[3]), &c, &s);
        float rdx = r * c, rdy = r * s;
        /* offset = u*rd.x + v*rd.y */
        offset = F3(fmaf(cam->v[0], rdy, cam->u[0] * rdx), fmaf(cam->v[1], rdy, cam->u[1] * rdx),
                    fmaf(cam->v[2], rdy, cam->u[2] * rdx));
    }
    f3 org = add3(ld3(cam->origin), offset);
    /* llc + s*horizontal + t*vertical - origin - offset */
    f3 d;
    d.x = fmaf(v, cam->vertical[0], fmaf(u, cam->horizontal[0], cam->lower_left_corner[0])) - cam->origin[0] - offset.x;
    d.y = fmaf(v, cam->vertical[1], fmaf(u, cam->horizontal[1], cam->lower_left_corner[1])) - cam->origin[1] - offset.y;
    d.z = fmaf(v, cam->vertical[2], fmaf(u, cam->horizontal[2], cam->lower_left_corner[2])) - cam->origin[2] - offset.z;
    float tm = cam->time0;
    if (cam->time0 != cam->time1) {
        uint32_t b1[4];
        rng_block(seed, (uint32_t)pixel, (uint32_t)sample, 1u, b1);
        tm = fmaf(cam->time1 - cam->time0, orc_u01(b1[0]), cam->time0);
    }
    st3(ray7, org);
    st3(ray7 + 3, d);
    ray7[6] = tm;
}

/* ------------------------------------------------------------------------------------------------
 * primitive tests.  Precision policy (DESIGN.md "precision"): the cancellation-prone part of the
 * sphere quadratic (oc, half_b, c, discriminant) is evaluated in double from the float inputs;
 * the roots are then formed in float with the cancellation-free pair q/a, c/q.
 * ---------------------------------------------------------------------------------------------- */
typedef struct { int type; /* 0 sphere 1 msphere 2 triangle 3 moving triangle */ int idx; } objref;

static inline objref obj_of(const orc_scene *s, int id)
{
    objref r;
    if (id < s->n_spheres) { r.type = 0; r.idx = id; }
    else if (id < s->n_spheres + s->n_mspheres) { r.type = 1; r.idx = id - s->n_spheres; }
    else if (id < s->n_spheres + s->n_mspheres + s->n_triangles) { r.type = 2; r.idx = id - s->n_spheres - s->n_mspheres; }
    else { r.type = 3; r.idx = id - s->n_spheres - s->n_mspheres - s->n_triangles; }
    return r;
}

/* sphere.h:33-58.  Accepts the nearest root in [t_min, t_max] (inclusive, as the reference). */
static int sphere_roots(f3 o, f3 d, f3 c, float radius, float t_min, float t_max, float *t_out)
{
    double ocx = (double)o.x - (double)c.x, ocy = (double)o.y - (double)c.y, ocz = (double)o.z - (double)c.z;
    double dx = d.x, dy = d.y, dz = d.z;
    double a = fma(dz, dz, fma(dy, dy, dx * dx));
    double hb = fma(ocz, dz, fma(ocy, dy, ocx * dx));
    double cc = fma(ocz, ocz, fma(ocy, ocy, ocx * ocx)) - (double)radius * (double)radius;
    double disc = fma(-a, cc, hb * hb);
    if (disc < 0.0) return 0;
    float sq = sqrtf((float)disc);
    float hbf = (float)hb, af = (float)a, ccf = (float)cc;
    float q = -(hbf + copysignf(sq, hbf));
    float r0 = q / af, r1 = ccf / q;
    float tn = fminf(r0, r1), tf = fmaxf(r0, r1);
    float root = tn;
    if (!(root >= t_min && root <= t_max)) {
        root = tf;
        if (!(root >= t_min && root <= t_max)) return 0;
    }
    *t_out = root;
    return 1;
}

/* moving_sphere.h:27-30 */
static inline f3 msphere_center(const rrtb_msphere *m, float time)
{
    float k = (time - m->time0) / (m->time1 - m->time0);
    return F3(fmaf(k, m->center1[0] - m->center0[0], m->center0[0]),
              fmaf(k, m->center1[1] - m->center0[1], m->center0[1]),
              fmaf(k, m->center1[2] - m->center0[2], m->center0[2]));
}

/* triangle.h:35-75 (Moeller-Trumbore).  Products are accumulated in double from the float inputs with
 * fixed fma chains; the barycentric tests are done on the numerators (no division):  with det = a,
 * u = un/det, v = vn/det the reference's  u<0 || u>1 || v<0 || u+v>1  is evaluated sign-aware.
 * t = float(tn) / float(det). */
static inline double dcross(double a, double b, double c, double d) { return fma(a, b, -(c * d)); } /* a*b - c*d */
static int triangle_t(f3 o, f3 d, double v0x, double v0y, double v0z, f3 e1f, f3 e2f, float t_min, float t_max, float *t_out)
{
    const double EPS = (double)1e-7f;
    double e1x = e1f.x, e1y = e1f.y, e1z = e1f.z, e2x = e2f.x, e2y = e2f.y, e2z = e2f.z;
    double dx = d.x, dy = d.y, dz = d.z;
    double hx = dcross(dy, e2z, dz, e2y), hy = dcross(dz, e2x, dx, e2z), hz = dcross(dx, e2y, dy, e2x);
    double det = fma(e1z, hz, fma(e1y, hy, e1x * hx));
    if (det > -EPS && det < EPS) return 0;
    double sx = (double)o.x - v0x, sy = (double)o.y - v0y, sz = (double)o.z - v0z;
    double un = fma(sz, hz, fma(sy, hy, sx * hx));
    double qx = dcross(sy, e1z, sz, e1y), qy = dcross(sz, e1x, sx, e1z), qz = dcross(sx, e1y, sy, e1x);
    double vn = fma(dz, qz, fma(dy, qy, dx * qx));
    if (det > 0.0) {
        if (un < 0.0 || un > det || vn < 0.0 || un + vn > det) return 0;
    }
    else {
        if (un > 0.0 || un < det || vn > 0.0 || un + vn < det) return 0;
    }
    double tn = fma(e2z, qz, fma(e2y, qy, e2x * qx));
    float t = (float)tn / (float)det;
    /* triangle.h:61 is exclusive at both ends; t == t_max (an exact tie with the current closest hit) is let
     * through here and settled by candidate_wins, which restates that exclusivity order-independently */
    if (t > 1e-7f && t > t_min && t <= t_max) {
        *t_out = t;
        return 1;
    }
    return 0;
}

/* triangle.h:9-15 */
static f3 triangle_normal(f3 v0, f3 v1, f3 v2)
{
    return unit3(cross3(unit3(sub3(v1, v0)), unit3(sub3(v2, v0))));
}

/* include/rrtb.h "rrtb_mtriangle": (base, rate) of v0, e1 = v1 - v0 and e2 = v2 - v0; a zero rate keeps its base exactly */
static void lin_of(float x_at_time0, float move, float dt, float time0, float *base, float *rate)
{
    *rate = move / dt;
    *base = *rate == 0.0f ? x_at_time0 : fmaf(-*rate, time0, x_at_time0);
}

void orc_mtriangle_record2(const rrtb_mtriangle *m, float base[3], float rate[3], float e1b[3], float e1r[3], float e2b[3], float e2r[3])
{
    float dt = m->time1 - m->time0;
    for (int k = 0; k < 3; ++k) {
        lin_of(m->v0[k], m->delta[k], dt, m->time0, &base[k], &rate[k]);
        lin_of(m->v1[k] - m->v0[k], m->extra1[k], dt, m->time0, &e1b[k], &e1r[k]);
        lin_of(m->v2[k] - m->v0[k], m->extra2[k], dt, m->time0, &e2b[k], &e2r[k]);
    }
}

/* the edges of the pose at `time` (float): e(t) = fma(rate, t, base); a zero rate keeps its base exactly */
static f3 edge_at(const float b[3], const float r[3], float time)
{
    return F3(r[0] == 0.0f ? b[0] : fmaf(r[0], time, b[0]), r[1] == 0.0f ? b[1] : fmaf(r[1], time, b[1]),
              r[2] == 0.0f ? b[2] : fmaf(r[2], time, b[2]));
}

void orc_mtriangle_record(const rrtb_mtriangle *m, float base[3], float rate[3], float e1[3], float e2[3])
{
    float e1r[3], e2r[3];
    orc_mtriangle_record2(m, base, rate, e1, e1r, e2, e2r); /* e1, e2 at time0-extrapolated-to-0: the bases */
}

void orc_triangle_normal(const rrtb_triangle *tr, float n[3])
{
    f3 v = triangle_normal(ld3(tr->v0), ld3(tr->v1), ld3(tr->v2));
    n[0] = v.x;
    n[1] = v.y;
    n[2] = v.z;
}

static int hit_t_only(const orc_scene *s, int id, f3 o, f3 d, float time, float t_min, float t_max, float *t)
{
    objref r = obj_of(s, id);
    if (r.type == 0) {
        const rrtb_sphere *sp = &s->spheres[r.idx];
        return sphere_roots(o, d, ld3(sp->center), sp->radius, t_min, t_max, t);
    }
    if (r.type == 1) {
        const rrtb_msphere *m = &s->mspheres[r.idx];
        return sphere_roots(o, d, msphere_center(m, time), m->radius, t_min, t_max, t);
    }
    if (r.type == 2) {
        const rrtb_triangle *tr = &s->triangles[r.idx];
        return triangle_t(o, d, (double)tr->v0[0], (double)tr->v0[1], (double)tr->v0[2], sub3(ld3(tr->v1), ld3(tr->v0)),
                          sub3(ld3(tr->v2), ld3(tr->v0)), t_min, t_max, t);
    }
    /* SURVEY 8f4: the instance moves, so the ray meets the triangle of the pose at its time: v0(time) in double from
     * the float (base, rate), the edges e1(time), e2(time) in float */
    float base[3], rate[3], e1b[3], e1r[3], e2b[3], e2r[3];
    orc_mtriangle_record2(&s->mtriangles[r.idx], base, rate, e1b, e1r, e2b, e2r);
    double tm = (double)time;
    return triangle_t(o, d, fma((double)rate[0], tm, (double)base[0]), fma((double)rate[1], tm, (double)base[1]),
                      fma((double)rate[2], tm, (double)base[2]), edge_at(e1b, e1r, time), edge_at(e2b, e2r, time), t_min, t_max, t);
}

/* hit_record fill: sphere.h:51-55, moving_sphere.h:51-55, triangle.h:62-66, hittable.h:16-20 */
static void hit_record_fill(const orc_scene *s, int id, f3 o, f3 d, float time, float t, float *rec7, int *mat)
{
    objref r = obj_of(s, id);
    f3 p = F3(fmaf(t, d.x, o.x), fmaf(t, d.y, o.y), fmaf(t, d.z, o.z));
    f3 n;
    if (r.type == 0) {
        const rrtb_sphere *sp = &s->spheres[r.idx];
        n = scl3(1.0f / sp->radius, sub3(p, ld3(sp->center)));
        *mat = sp->material;
    }
    else if (r.type == 1) {
        const rrtb_msphere *m = &s->mspheres[r.idx];
        n = scl3(1.0f / m->radius, sub3(p, msphere_center(m, time)));
        *mat = m->material;
    }
    else if (r.type == 2) {
        const rrtb_triangle *tr = &s->triangles[r.idx];
        n = triangle_normal(ld3(tr->v0), ld3(tr->v1), ld3(tr->v2));
        *mat = tr->material;
    }
    else { /* the face normal of the pose at the ray's time: unit(cross(unit(e1), unit(e2))), triangle.h:9-15 */
        const rrtb_mtriangle *m = &s->mtriangles[r.idx];
        float base[3], rate[3], e1b[3], e1r[3], e2b[3], e2r[3];
        orc_mtriangle_record2(m, base, rate, e1b, e1r, e2b, e2r);
        n = unit3(cross3(unit3(edge_at(e1b, e1r, time)), unit3(edge_at(e2b, e2r, time))));
        *mat = m->material;
    }
    int front = dot3(d, n) < 0.0f;
    if (!front) n = F3(-n.x, -n.y, -n.z);
    st3(rec7, p);
    st3(rec7 + 3, n);
    rec7[6] = front ? 1.0f : 0.0f;
}

int orc_hit_object(const orc_scene *s, int id, const float *ray7, float t_min, float t_max, float *t, float *rec7)
{
    f3 o = ld3(ray7), d = ld3(ray7 + 3);
    float tt;
    if (!hit_t_only(s, id, o, d, ray7[6], t_min, t_max, &tt)) return 0;
    *t = tt;
    if (rec7) {
        int mat;
        hit_record_fill(s, id, o, d, ray7[6], tt, rec7, &mat);
    }
    return 1;
}

/* The order-independent restatement of the scan's tie rule (hittable_list.h:102-114 with the
 * inclusive sphere test sphere.h:45-48 and the exclusive triangle test triangle.h:61): among
 * candidates at exactly equal t the last sphere-like object in id order wins, else the first
 * triangle.  Expressed as "does candidate (t,id) beat current best (bt,bid)". */
static inline int is_tri(const orc_scene *s, int id) { return id >= s->n_spheres + s->n_mspheres; }
static inline int candidate_wins(const orc_scene *s, float t, int id, float bt, int bid)
{
    if (bid < 0) return 1;
    if (t < bt) return 1;
    if (t > bt) return 0;
    int ct = is_tri(s, id), bt_tri = is_tri(s, bid);
    if (ct != bt_tri) return !ct;     /* sphere-like beats triangle */
    return ct ? (id < bid) : (id > bid);
}

static int closest_scan(const orc_scene *s, f3 o, f3 d, float time, float t_min, float *t_out, orc_counters *cnt)
{
    int n = orc_n_objects(s);
    float best = INFINITY;
    int bid = -1;
    for (int id = 0; id < n; ++id) {
        float t;
        if (hit_t_only(s, id, o, d, time, t_min, best, &t) && candidate_wins(s, t, id, best, bid)) {
            best = t;
            bid = id;
        }
    }
    if (cnt) {
        cnt->sphere_tests += (uint64_t)s->n_spheres;
        cnt->msphere_tests += (uint64_t)s->n_mspheres;
        cnt->triangle_tests += (uint64_t)s->n_triangles + (uint64_t)s->n_mtriangles;
    }
    *t_out = best;
    return bid;
}

void orc_trace_scan(const orc_scene *s, const float *rays7, int n, float t_min, int32_t *id, float *t, float *rec7)
{
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; ++i) {
        const float *r = rays7 + 7 * (size_t)i;
        float tt;
        int b = closest_scan(s, ld3(r), ld3(r + 3), r[6], t_min, &tt, NULL);
        id[i] = b;
        t[i] = b >= 0 ? tt : -1.0f;
        if (rec7) {
            float *o = rec7 + 7 * (size_t)i;
            memset(o, 0, 7 * sizeof(float));
            int mat;
            if (b >= 0) hit_record_fill(s, b, ld3(r), ld3(r + 3), r[6], tt, o, &mat);
        }
    }
}

/* ------------------------------------------------------------------------------------------------
 * canonical LBVH (SURVEY Appendix D): boxes as sphere.h:60-64, moving_sphere.h:60-66 (shutter
 * union, bvh.h:152), triangle.h:77-87; Morton codes; stable sort on (code, id); Karras 2012;
 * bottom-up refit with fminf/fmaxf.
 * ---------------------------------------------------------------------------------------------- */
static void prim_box(const orc_scene *s, int id, float *b)
{
    objref r = obj_of(s, id);
    if (r.type == 0) {
        const rrtb_sphere *sp = &s->spheres[r.idx];
        for (int k = 0; k < 3; ++k) {
            /* sphere.h:60-64 with |radius|: the reference's center -+ radius is an INVERTED box for the negative radii the
             * book uses for hollow glass, and its bvh then loses the sphere; equal to the reference for radius >= 0 */
            b[k] = sp->center[k] - fabsf(sp->radius);
            b[3 + k] = sp->center[k] + fabsf(sp->radius);
        }
    }
    else if (r.type == 1) {
        const rrtb_msphere *m = &s->mspheres[r.idx];
        /* center(time) = c0 + ((time - t0)/(t1 - t0)) * (c1 - c0), mul then add (moving_sphere.h:27-30) */
        float k0 = (s->cam.time0 - m->time0) / (m->time1 - m->time0);
        float k1 = (s->cam.time1 - m->time0) / (m->time1 - m->time0);
        for (int k = 0; k < 3; ++k) {
            float dc = m->center1[k] - m->center0[k];
            float ca = m->center0[k] + k0 * dc;
            float cb = m->center0[k] + k1 * dc;
            b[k] = fminf(ca - fabsf(m->radius), cb - fabsf(m->radius));
            b[3 + k] = fmaxf(ca + fabsf(m->radius), cb + fabsf(m->radius));
        }
    }
    else if (r.type == 2) {
        const rrtb_triangle *t = &s->triangles[r.idx];
        for (int k = 0; k < 3; ++k) {
            b[k] = fminf(fminf(t->v0[k], t->v1[k]), t->v2[k]);
            b[3 + k] = fmaxf(fmaxf(t->v0[k], t->v1[k]), t->v2[k]);
        }
    }
    else { /* union of the poses at the two ends of the shutter, T = camera time0 / time1: {v0(T), v0(T)+e1(T), v0(T)+e2(T)};
            * motion is linear in time, so they bound every pose in between */
        float base[3], rate[3], e1b[3], e1r[3], e2b[3], e2r[3];
        orc_mtriangle_record2(&s->mtriangles[r.idx], base, rate, e1b, e1r, e2b, e2r);
        f3 ea1 = edge_at(e1b, e1r, s->cam.time0), ea2 = edge_at(e2b, e2r, s->cam.time0);
        f3 eb1 = edge_at(e1b, e1r, s->cam.time1), eb2 = edge_at(e2b, e2r, s->cam.time1);
        const float a1[3] = {ea1.x, ea1.y, ea1.z}, a2[3] = {ea2.x, ea2.y, ea2.z}, b1[3] = {eb1.x, eb1.y, eb1.z}, b2[3] = {eb2.x, eb2.y, eb2.z};
        for (int k = 0; k < 3; ++k) {
            float pa = fmaf(rate[k], s->cam.time0, base[k]), pb = fmaf(rate[k], s->cam.time1, base[k]);
            float lo = fminf(fminf(fminf(pa, pa + a1[k]), pa + a2[k]), fminf(fminf(pb, pb + b1[k]), pb + b2[k]));
            float hi = fmaxf(fmaxf(fmaxf(pa, pa + a1[k]), pa + a2[k]), fmaxf(fmaxf(pb, pb + b1[k]), pb + b2[k]));
            b[k] = lo;
            b[3 + k] = hi;
        }
    }
}

static inline uint32_t expand_bits10(uint32_t v)
{
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

static inline int clz64(uint64_t x) { return x ? __builtin_clzll(x) : 64; }

static inline int delta_fn(const uint64_t *keys, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    return clz64(keys[i] ^ keys[j]);
}

static int cmp_u64(const void *a, const void *b)
{
    uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
    return x < y ? -1 : (x > y ? 1 : 0);
}

orc_bvh *orc_bvh_build(const orc_scene *s)
{
    int n = orc_n_objects(s);
    orc_bvh *b = (orc_bvh *)calloc(1, sizeof(orc_bvh));
    b->n = n;
    b->morton = (uint32_t *)calloc((size_t)n, 4);
    b->perm = (uint32_t *)calloc((size_t)n, 4);
    int ni = n > 1 ? n - 1 : 0;
    b->left = (int32_t *)calloc((size_t)(ni ? ni : 1), 4);
    b->right = (int32_t *)calloc((size_t)(ni ? ni : 1), 4);
    b->parent = (int32_t *)calloc((size_t)(2 * n), 4);
    b->node_box = (float *)calloc((size_t)(6 * (ni ? ni : 1)), 4);
    b->prim_box = (float *)calloc((size_t)(6 * n), 4);

    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    float mag = 0.0f;
    float *cent = (float *)malloc((size_t)n * 3 * sizeof(float));
    for (int i = 0; i < n; ++i) {
        float *pb = b->prim_box + 6 * (size_t)i;
        prim_box(s, i, pb);
        for (int k = 0; k < 3; ++k) {
            float c = 0.5f * (pb[k] + pb[3 + k]);
            cent[3 * (size_t)i + k] = c;
            lo[k] = fminf(lo[k], c);
            hi[k] = fmaxf(hi[k], c);
            mag = fmaxf(mag, fmaxf(fabsf(pb[k]), fabsf(pb[3 + k])));
        }
    }
    for (int k = 0; k < 3; ++k) mag = fmaxf(mag, fabsf(s->cam.origin[k]) + s->cam.lens_radius);
    b->pad = mag * 9.5367431640625e-07f; /* 2^-20 * largest coordinate magnitude (DESIGN.md "box padding") */

    float inv[3];
    for (int k = 0; k < 3; ++k) {
        float ext = hi[k] - lo[k];
        inv[k] = ext > 0.0f ? 1.0f / ext : 0.0f;
    }
    uint64_t *keys = (uint64_t *)malloc((size_t)n * 8);
    for (int i = 0; i < n; ++i) {
        uint32_t q[3];
        for (int k = 0; k < 3; ++k) {
            float x = (cent[3 * (size_t)i + k] - lo[k]) * inv[k];
            int v = (int)(x * 1024.0f);
            v = v < 0 ? 0 : (v > 1023 ? 1023 : v);
            q[k] = (uint32_t)v;
        }
        uint32_t code = (expand_bits10(q[0]) << 2) | (expand_bits10(q[1]) << 1) | expand_bits10(q[2]);
        b->morton[i] = code;
        keys[i] = ((uint64_t)code << 32) | (uint32_t)i;
    }
    free(cent);
    qsort(keys, (size_t)n, 8, cmp_u64); /* keys are unique, so any correct sort gives this order */
    for (int k = 0; k < n; ++k) b->perm[k] = (uint32_t)keys[k];

    for (int i = 0; i < 2 * n - 1; ++i) b->parent[i] = -1;
    for (int i = 0; i < ni; ++i) {
        int d = (delta_fn(keys, n, i, i + 1) - delta_fn(keys, n, i, i - 1)) >= 0 ? 1 : -1;
        int dmin = delta_fn(keys, n, i, i - d);
        int lmax = 2;
        while (delta_fn(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
        int l = 0;
        for (int t = lmax / 2; t >= 1; t /= 2)
            if (delta_fn(keys, n, i, i + (l + t) * d) > dmin) l += t;
        int j = i + l * d;
        int dnode = delta_fn(keys, n, i, j);
        int sp = 0;
        int t = l;
        do {
            t = (t + 1) >> 1;
            if (delta_fn(keys, n, i, i + (sp + t) * d) > dnode) sp += t;
        } while (t > 1);
        int gamma = i + sp * d + (d < 0 ? -1 : 0);
        int mn = i < j ? i : j, mx = i < j ? j : i;
        int32_t L = (mn == gamma) ? ~gamma : gamma;
        int32_t R = (mx == gamma + 1) ? ~(gamma + 1) : gamma + 1;
        b->left[i] = L;
        b->right[i] = R;
        b->parent[L >= 0 ? L : (ni + ~L)] = i;
        b->parent[R >= 0 ? R : (ni + ~R)] = i;
    }
    free(keys);

    /* refit: bottom-up from every leaf, second arrival computes the box */
    if (ni > 0) {
        int *visits = (int *)calloc((size_t)ni, sizeof(int));
        for (int k = 0; k < n; ++k) {
            int node = b->parent[ni + k];
            while (node >= 0) {
                if (++visits[node] < 2) break;
                float *nb = b->node_box + 6 * (size_t)node;
                const float *lb = b->left[node] >= 0 ? b->node_box + 6 * (size_t)b->left[node]
                                                     : b->prim_box + 6 * (size_t)b->perm[~b->left[node]];
                const float *rb = b->right[node] >= 0 ? b->node_box + 6 * (size_t)b->right[node]
                                                      : b->prim_box + 6 * (size_t)b->perm[~b->right[node]];
                for (int c = 0; c < 3; ++c) {
                    nb[c] = fminf(lb[c], rb[c]);
                    nb[3 + c] = fmaxf(lb[3 + c], rb[3 + c]);
                }
                node = b->parent[node];
            }
        }
        free(visits);
    }
    return b;
}

void orc_bvh_free(orc_bvh *b)
{
    if (!b) return;
    free(b->morton); free(b->perm); free(b->left); free(b->right); free(b->parent);
    free(b->node_box); free(b->prim_box); free(b);
}

/* aabb.h:18-93 restated with precomputed reciprocal direction (one FMA per plane) on a box padded
 * by bvh->pad; the test is inclusive so it can only over-accept relative to the reference. */
static inline int box_hit(const float *bx, float pad, f3 inv, f3 ood, float t_min, float t_max)
{
    float x0 = fmaf(bx[0] - pad, inv.x, ood.x), x1 = fmaf(bx[3] + pad, inv.x, ood.x);
    float y0 = fmaf(bx[1] - pad, inv.y, ood.y), y1 = fmaf(bx[4] + pad, inv.y, ood.y);
    float z0 = fmaf(bx[2] - pad, inv.z, ood.z), z1 = fmaf(bx[5] + pad, inv.z, ood.z);
    float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), t_min));
    float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), t_max));
    return tn <= tf;
}

static int closest_bvh(const orc_scene *s, const orc_bvh *b, f3 o, f3 d, float time, float t_min, float *t_out,
                       orc_counters *cnt)
{
    float best = INFINITY;
    int bid = -1;
    int n = b->n;
    if (n == 0) { *t_out = best; return -1; }
    if (n == 1) {
        float t;
        if (hit_t_only(s, 0, o, d, time, t_min, best, &t)) { best = t; bid = 0; }
        *t_out = best;
        return bid;
    }
    /* direction components of (almost) exactly zero would make the FMA-form slab test compute inf - inf */
    f3 ds = F3(fabsf(d.x) < 1e-20f ? copysignf(1e-20f, d.x) : d.x, fabsf(d.y) < 1e-20f ? copysignf(1e-20f, d.y) : d.y,
               fabsf(d.z) < 1e-20f ? copysignf(1e-20f, d.z) : d.z);
    f3 inv = F3(1.0f / ds.x, 1.0f / ds.y, 1.0f / ds.z);
    f3 ood = F3(-o.x * inv.x, -o.y * inv.y, -o.z * inv.z);
    int32_t stack[128];
    int sp = 0;
    stack[sp++] = 0;
    if (cnt) cnt->box_tests++;
    if (!box_hit(b->node_box, b->pad, inv, ood, t_min, best)) { *t_out = best; return -1; }
    while (sp > 0) {
        int32_t node = stack[--sp];
        int32_t ch[2] = {b->left[node], b->right[node]};
        for (int c = 0; c < 2; ++c) {
            int32_t k = ch[c];
            const float *bx = k >= 0 ? b->node_box + 6 * (size_t)k : b->prim_box + 6 * (size_t)b->perm[~k];
            if (cnt) cnt->box_tests++;
            if (!box_hit(bx, b->pad, inv, ood, t_min, best)) continue;
            if (k >= 0) {
                stack[sp++] = k;
            }
            else {
                int id = (int)b->perm[~k];
                float t;
                if (cnt) {
                    if (id < s->n_spheres) cnt->sphere_tests++;
                    else if (id < s->n_spheres + s->n_mspheres) cnt->msphere_tests++;
                    else cnt->triangle_tests++;
                }
                if (hit_t_only(s, id, o, d, time, t_min, best, &t) && candidate_wins(s, t, id, best, bid)) {
                    best = t;
                    bid = id;
                }
            }
        }
    }
    *t_out = best;
    return bid;
}

void orc_trace_bvh(const orc_scene *s, const orc_bvh *b, const float *rays7, int n, float t_min, int32_t *id,
                   float *t, float *rec7, orc_counters *cnt)
{
    orc_counters total;
    memset(&total, 0, sizeof(total));
#pragma omp parallel
    {
        orc_counters local;
        memset(&local, 0, sizeof(local));
#pragma omp for schedule(static)
        for (int i = 0; i < n; ++i) {
            const float *r = rays7 + 7 * (size_t)i;
            float tt;
            int bid = closest_bvh(s, b, ld3(r), ld3(r + 3), r[6], t_min, &tt, &local);
            local.rays++;
            if (bid >= 0) local.hits++;
            id[i] = bid;
            t[i] = bid >= 0 ? tt : -1.0f;
            if (rec7) {
                float *o = rec7 + 7 * (size_t)i;
                memset(o, 0, 7 * sizeof(float));
                int mat;
                if (bid >= 0) hit_record_fill(s, bid, ld3(r), ld3(r + 3), r[6], tt, o, &mat);
            }
        }
#pragma omp critical
        {
            total.rays += local.rays; total.hits += local.hits; total.box_tests += local.box_tests;
            total.sphere_tests += local.sphere_tests; total.msphere_tests += local.msphere_tests;
            total.triangle_tests += local.triangle_tests;
        }
    }
    if (cnt) *cnt = total;
}

/* ------------------------------------------------------------------------------------------------
 * materials (material.h).  One Philox block per bounce:
 *   x0,x1 -> direction on the unit sphere (z = 1-2*x0, phi = 2*pi*x1)   [lambertian, metal fuzz]
 *   x2 and the two 16-bit halves of word 3 -> ball radius = max of three uniforms (pdf 3r^2) [metal]
 *   x0 -> reflect/refract choice                                         [dielectric]
 * Distributions equal the reference's rejection samplers (vec3.h:127-145); only the mapping from
 * random numbers to samples differs, which the reference's own RNG change (CPU mt19937 vs GPU
 * XORWOW) already does.
 * ---------------------------------------------------------------------------------------------- */
static f3 sample_unit_sphere(float x0, float x1)
{
    float z = fmaf(-2.0f, x0, 1.0f);
    float r = sqrtf(fmaxf(0.0f, fmaf(-z, z, 1.0f)));
    float c, s;
    orc_sincos2pi(x1, &c, &s);
    return F3(r * c, r * s, z);
}

/* returns 1 if the path continues; dir/atten out */
static int scatter_one(const rrtb_material *m, f3 d_in, f3 n, int front, const uint32_t rnd[4], f3 *dir, f3 *att)
{
    if (m->type == RRTB_DIFFUSE_LIGHT) { /* book 2 diffuse_light: never scatters; att = Le */
        *dir = F3(0.0f, 0.0f, 0.0f);
        *att = ld3(m->albedo);
        return 0;
    }
    if (m->type == RRTB_LAMBERTIAN) { /* material.h:21-32 */
        f3 u = sample_unit_sphere(orc_u01(rnd[0]), orc_u01(rnd[1]));
        f3 sd = add3(n, u);
        if (fabsf(sd.x) < 1e-8f && fabsf(sd.y) < 1e-8f && fabsf(sd.z) < 1e-8f) sd = n;
        *dir = sd;
        *att = ld3(m->albedo);
        return 1;
    }
    if (m->type == RRTB_METAL) { /* material.h:48-57 */
        f3 ud = unit3(d_in);
        float dn = dot3(ud, n);
        f3 refl = F3(fmaf(-2.0f * dn, n.x, ud.x), fmaf(-2.0f * dn, n.y, ud.y), fmaf(-2.0f * dn, n.z, ud.z));
        float fuzz = fabsf(m->param < 1.0f ? m->param : 1.0f); /* fuzz * random_in_unit_sphere(): radius |fuzz| */
        if (fuzz > 0.0f) {
            f3 u = sample_unit_sphere(orc_u01(rnd[0]), orc_u01(rnd[1]));
            float ra = orc_u01(rnd[2]);
            float rb = (float)(rnd[3] >> 16) * 1.52587890625e-05f;
            float rc = (float)(rnd[3] & 0xFFFFu) * 1.52587890625e-05f;
            float rad = fmaxf(ra, fmaxf(rb, rc)) * fuzz;
            refl = F3(fmaf(rad, u.x, refl.x), fmaf(rad, u.y, refl.y), fmaf(rad, u.z, refl.z));
        }
        *dir = refl;
        *att = ld3(m->albedo);
        return dot3(refl, n) > 0.0f;
    }
    /* dielectric, material.h:76-109 */
    float ir = m->param;
    float eta = front ? 1.0f / ir : ir;
    f3 ud = unit3(d_in);
    float cos_t = fminf(-dot3(ud, n), 1.0f);
    float sin_t = sqrtf(fmaxf(0.0f, fmaf(-cos_t, cos_t, 1.0f)));
    int cannot = eta * sin_t > 1.0f;
    float r0 = (1.0f - eta) / (1.0f + eta);
    r0 = r0 * r0;
    float om = 1.0f - cos_t;
    float om2 = om * om;
    float refl_p = fmaf(1.0f - r0, om2 * om2 * om, r0);
    if (cannot || refl_p > orc_u01(rnd[0])) {
        float dn = dot3(ud, n);
        *dir = F3(fmaf(-2.0f * dn, n.x, ud.x), fmaf(-2.0f * dn, n.y, ud.y), fmaf(-2.0f * dn, n.z, ud.z));
    }
    else { /* vec3.h:158-164 */
        f3 perp = scl3(eta, F3(fmaf(cos_t, n.x, ud.x), fmaf(cos_t, n.y, ud.y), fmaf(cos_t, n.z, ud.z)));
        float k = -sqrtf(fabsf(1.0f - dot3(perp, perp)));
        *dir = F3(fmaf(k, n.x, perp.x), fmaf(k, n.y, perp.y), fmaf(k, n.z, perp.z));
    }
    *att = F3(1.0f, 1.0f, 1.0f);
    return 1;
}

void orc_scatter(const orc_scene *s, const float *in16, const uint32_t *rnd4, int n, float *out8)
{
    for (int i = 0; i < n; ++i) {
        const float *in = in16 + 16 * (size_t)i;
        float *o = out8 + 8 * (size_t)i;
        f3 dir, att;
        int mat = (int)in[14];
        int ok = scatter_one(&s->materials[mat], ld3(in + 3), ld3(in + 10), in[13] != 0.0f, rnd4 + 4 * (size_t)i,
                             &dir, &att);
        st3(o, dir);
        st3(o + 3, att);
        o[6] = ok ? 1.0f : 0.0f;
        o[7] = 0.0f;
    }
}

/* ------------------------------------------------------------------------------------------------
 * the estimator: rrt.cu:42-79 (ray_color) and rrt.cu:109-121 (per-pixel sample loop)
 * ---------------------------------------------------------------------------------------------- */
void orc_path(const orc_scene *s, const orc_bvh *bvh, int W, int H, int pixel, int sample, int max_depth,
              uint64_t seed, float *rgb, orc_counters *cnt)
{
    float ray7[7];
    orc_camera_ray(&s->cam, W, H, pixel, sample, seed, ray7);
    orc_radiance(s, bvh, ray7, pixel, sample, max_depth, seed, rgb, cnt);
}

/* ray_color (rrt.cu:42-79) for an explicit primary ray; (pixel, sample) only key the bounce RNG.  bg: the constant
 * background that replaces the sky, or NULL for the sky */
static void radiance(const orc_scene *s, const float *bg, const orc_bvh *bvh, const float *ray7, int pixel, int sample,
                     int max_depth, uint64_t seed, float *rgb, orc_counters *cnt)
{
    f3 o = ld3(ray7), d = ld3(ray7 + 3);
    float time = ray7[6];
    f3 thr = F3(1.f, 1.f, 1.f);
    rgb[0] = rgb[1] = rgb[2] = 0.0f;
    if (cnt) cnt->paths++;
    for (int b = 0; b < max_depth; ++b) {
        float t;
        int id = bvh ? closest_bvh(s, bvh, o, d, time, 0.001f, &t, cnt) : closest_scan(s, o, d, time, 0.001f, &t, cnt);
        if (cnt) cnt->rays++;
        if (id < 0 && bg) {
            rgb[0] = thr.x * bg[0];
            rgb[1] = thr.y * bg[1];
            rgb[2] = thr.z * bg[2];
            return;
        }
        if (id < 0) { /* sky, rrt.cu:68-75 */
            float uy = d.y * (1.0f / sqrtf(dot3(d, d)));
            float tt = 0.5f * (uy + 1.0f);
            f3 c = F3(fmaf(tt, 0.5f, 1.0f - tt), fmaf(tt, 0.7f, 1.0f - tt), fmaf(tt, 1.0f, 1.0f - tt));
            rgb[0] = thr.x * c.x;
            rgb[1] = thr.y * c.y;
            rgb[2] = thr.z * c.z;
            return;
        }
        if (cnt) cnt->hits++;
        float rec[7];
        int mat;
        hit_record_fill(s, id, o, d, time, t, rec, &mat);
        uint32_t rnd[4];
        rng_block(seed, (uint32_t)pixel, (uint32_t)sample, 2u + (uint32_t)b, rnd);
        f3 dir, att;
        if (!scatter_one(&s->materials[mat], d, ld3(rec + 3), rec[6] != 0.0f, rnd, &dir, &att)) {
            if (s->materials[mat].type == RRTB_DIFFUSE_LIGHT) { /* emitter: throughput x Le (att = Le) */
                rgb[0] = thr.x * att.x;
                rgb[1] = thr.y * att.y;
                rgb[2] = thr.z * att.z;
            }
            return; /* else absorbed: black */
        }
        thr = F3(thr.x * att.x, thr.y * att.y, thr.z * att.z);
        o = ld3(rec);
        d = dir;
    }
    /* exceeded depth: black (rrt.cu:78) */
}

void orc_radiance(const orc_scene *s, const orc_bvh *bvh, const float *ray7, int pixel, int sample, int max_depth,
                  uint64_t seed, float *rgb, orc_counters *cnt)
{
    radiance(s, NULL, bvh, ray7, pixel, sample, max_depth, seed, rgb, cnt);
}

static inline uint64_t to_fixed(float x, float clamp) /* value * 2^40, round to nearest even, clamped to [0, clamp] */
{
    if (!(x > 0.0f)) return 0;
    if (x > clamp) x = clamp;
    return (uint64_t)llrint((double)x * 1099511627776.0);
}

void orc_render(const orc_scene *s, const orc_bvh *bvh, int W, int H, int spp, int max_depth, uint64_t seed,
                int rank, int world, int shard_mode, float *out_rgb, uint64_t *out_fixed, orc_counters *cnt)
{
    orc_render_bg(s, NULL, bvh, W, H, spp, max_depth, seed, rank, world, shard_mode, out_rgb, out_fixed, cnt);
}

void orc_render_bg(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                   uint64_t seed, int rank, int world, int shard_mode, float *out_rgb, uint64_t *out_fixed,
                   orc_counters *cnt)
{
    orc_counters total;
    memset(&total, 0, sizeof(total));
    int tiles_x = (W + 7) / 8;
    const float clamp = orc_fixed_clamp(spp); /* the total spp: every shard clamps alike */
    if (world < 1) world = 1;
#pragma omp parallel
    {
        orc_counters local;
        memset(&local, 0, sizeof(local));
#pragma omp for schedule(dynamic, 4)
        for (int j = 0; j < H; ++j) {
            for (int i = 0; i < W; ++i) {
                int pixel = j * W + i;
                uint64_t acc[3] = {0, 0, 0};
                int mine = 1;
                if (world > 1 && shard_mode == RRTB_SHARD_TILES) {
                    int tile = (j / 4) * tiles_x + (i / 8);
                    mine = (tile % world) == rank;
                }
                if (mine) {
                    for (int sm = 0; sm < spp; ++sm) {
                        if (world > 1 && shard_mode == RRTB_SHARD_SAMPLES && (sm % world) != rank) continue;
                        float ray7[7], rgb[3];
                        orc_camera_ray(&s->cam, W, H, pixel, sm, seed, ray7);
                        radiance(s, bg, bvh, ray7, pixel, sm, max_depth, seed, rgb, &local);
                        for (int k = 0; k < 3; ++k) acc[k] += to_fixed(rgb[k], clamp);
                    }
                }
                for (int k = 0; k < 3; ++k) {
                    if (out_fixed) out_fixed[3 * (size_t)pixel + k] = acc[k];
                    if (out_rgb) out_rgb[3 * (size_t)pixel + k] = (float)((double)acc[k] * 9.094947017729282e-13);
                }
            }
        }
#pragma omp critical
        {
            total.rays += local.rays; total.hits += local.hits; total.box_tests += local.box_tests;
            total.sphere_tests += local.sphere_tests; total.msphere_tests += local.msphere_tests;
            total.triangle_tests += local.triangle_tests; total.paths += local.paths;
        }
    }
    if (cnt) *cnt = total;
}

/* color.h:8-23 and the flip of main.cpp:150-163 */
void orc_tonemap_rgb8(const float *rgb_sum, int W, int H, int spp, uint8_t *rgb8)
{
    float scale = 1.0f / (float)spp;
    for (int j = H - 1, k = 0; j >= 0; --j, ++k) {
        for (int i = 0; i < W; ++i) {
            for (int c = 0; c < 3; ++c) {
                float x = sqrtf(scale * rgb_sum[3 * ((size_t)j * W + i) + c]);
                /* clamp() returns double (rtweekend.h:93-98): 256 * clamp(...) is a double product */
                double cl = x < 0.0f ? 0.0 : (x > 0.999f ? (double)0.999f : (double)x);
                rgb8[3 * ((size_t)k * W + i) + c] = (uint8_t)(int)(256 * cl);
            }
        }
    }
}
