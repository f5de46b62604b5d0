/* rrt_oracle_f64.c -- TEST INFRASTRUCTURE ONLY: CPU oracle of the DOUBLE-precision integrator (SURVEY 8f1).
 *
 * What the reference's `rrtd` / `rrto` builds compute (FP_T = double, rtweekend.h:20-28), restated in plain C
 * over the float-rounded scene the C ABI carries ("double arithmetic on identical inputs"), with the product's
 * Philox streams and direct samplers.  Same rules as rrt_oracle.c: only tests/, smoke() and bench.py's
 * cpu_baseline leg may load it; every operation is one IEEE rounding (-ffp-contract=off, explicit fma()).
 * Pinned against oracle/_ref/libref_d.so in tests/test_f64_oracle.py.
 */
#include <math.h>
#include <string.h>

#include "rrt_oracle.h"

typedef struct { double x, y, z; } d3;
static inline d3 D3(double x, double y, double z) { d3 r = {x, y, z}; return r; }
static inline d3 ldf(const float *p) { return D3(p[0], p[1], p[2]); }
static inline d3 ldd(const double *p) { return D3(p[0], p[1], p[2]); }
static inline void std3(double *p, d3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
static inline d3 dsub(d3 a, d3 b) { return D3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline double ddot(d3 a, d3 b) { return fma(a.z, b.z, fma(a.y, b.y, a.x * b.x)); }
static inline double dcr(double a, double b, double c, double d) { return fma(a, b, -(c * d)); }

static inline double u01d(uint32_t x) { return (double)(x >> 8) * 5.9604644775390625e-08; }

static void rng_block(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t dim, uint32_t out[4])
{
    uint32_t ctr[4] = {pixel, sample, dim, 0u};
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    orc_philox4x32_10(ctr, key, out);
}

/* the float oracle's quadrant-exact polynomial, evaluated in double (sampling needs no more accuracy) */
static void sincos2pi_d(double u, double *c, double *s)
{
    double x = u - 0.5;
    double qf = rint(x * 4.0);
    double r = fma(qf, -0.25, x);
    double a = r * 6.283185307179586;
    double a2 = a * a;
    double sp = fma(a2, -1.9515295891e-4, 8.3321608736e-3);
    sp = fma(a2, sp, -1.6666654611e-1);
    double sn = fma(a * a2, sp, a);
    double cp = fma(a2, 2.443315711809948e-5, -1.388731625493765e-3);
    cp = fma(a2, cp, 4.166664568298827e-2);
    cp = fma(a2, cp, -0.5);
    double cs = fma(a2, cp, 1.0);
    int q = (int)qf & 3;
    double co = (q & 1) ? sn : cs, si = (q & 1) ? cs : sn;
    if (q == 1 || q == 2) co = -co;
    if (q >= 2) si = -si;
    *c = co;
    *s = si;
}

/* rrt.cu:112-114 + camera.h:31-38 in double.  ray7 = o(3) d(3) time */
void orc_d_camera_ray(const rrtb_camera *cam, int W, int H, int pixel, int sample, uint64_t seed, double *ray7)
{
    uint32_t b0[4];
    rng_block(seed, (uint32_t)pixel, (uint32_t)sample, 0u, b0);
    int i = pixel % W, j = pixel / W;
    double u = ((double)i + u01d(b0[0])) / (double)(W - 1);
    double v = ((double)j + u01d(b0[1])) / (double)(H - 1);
    d3 off = D3(0, 0, 0);
    if (cam->lens_radius > 0.0f) {
        double r = sqrt(u01d(b0[2])) * (double)cam->lens_radius;
        double c, s;
        sincos2pi_d(u01d(b0[3]), &c, &s);
        double rdx = r * c, rdy = r * s;
        off = D3(fma((double)cam->v[0], rdy, (double)cam->u[0] * rdx), fma((double)cam->v[1], rdy, (double)cam->u[1] * rdx),
                 fma((double)cam->v[2], rdy, (double)cam->u[2] * rdx));
    }
    for (int k = 0; k < 3; ++k) {
        double o = (double)cam->origin[k], of = k == 0 ? off.x : (k == 1 ? off.y : off.z);
        ray7[k] = o + of;
        ray7[3 + k] = fma(v, (double)cam->vertical[k], fma(u, (double)cam->horizontal[k], (double)cam->lower_left_corner[k])) - o - of;
    }
    double tm = cam->time0;
    if (cam->time0 != cam->time1) {
        uint32_t b1[4];
        rng_block(seed, (uint32_t)pixel, (uint32_t)sample, 1u, b1);
        tm = fma((double)cam->time1 - (double)cam->time0, u01d(b1[0]), (double)cam->time0);
    }
    ray7[6] = tm;
}

/* sphere.h:33-58 in double; the roots through the cancellation-free pair q/a, c/q */
static int sphere_d(d3 o, d3 d, d3 c, double rad, double t_min, double t_max, double *t_out)
{
    d3 oc = dsub(o, c);
    double a = ddot(d, d), hb = ddot(oc, d);
    double cc = fma(-rad, rad, ddot(oc, oc));
    double disc = fma(-a, cc, hb * hb);
    if (disc < 0.0) return 0;
    double sq = sqrt(disc);
    double q = -(hb + copysign(sq, hb));
    double r0 = q / a, r1 = cc / q;
    double tn = fmin(r0, r1), tf = fmax(r0, r1);
    double root = tn;
    if (!(root >= t_min && root <= t_max)) {
        root = tf;
        if (!(root >= t_min && root <= t_max)) return 0;
    }
    *t_out = root;
    return 1;
}

/* moving_sphere.h:27-30 on the product's leaf record: c0 + k * float(c1 - c0), k = (time - t0) / float(t1 - t0) */
static d3 msphere_center_d(const rrtb_msphere *m, double time)
{
    float dt = m->time1 - m->time0;
    float dc[3] = {m->center1[0] - m->center0[0], m->center1[1] - m->center0[1], m->center1[2] - m->center0[2]};
    double k = (time - (double)m->time0) / (double)dt;
    return D3(fma(k, (double)dc[0], (double)m->center0[0]), fma(k, (double)dc[1], (double)m->center0[1]),
              fma(k, (double)dc[2], (double)m->center0[2]));
}

/* triangle.h:35-75 in double; edges from the float-rounded e1, e2 the product stores */
static int triangle_d(d3 o, d3 d, d3 v0, const float e1f[3], const float e2f[3], double t_min, double t_max, double *t_out)
{
    const double EPS = 1e-7;
    d3 e1 = ldf(e1f), e2 = ldf(e2f);
    d3 h = D3(dcr(d.y, e2.z, d.z, e2.y), dcr(d.z, e2.x, d.x, e2.z), dcr(d.x, e2.y, d.y, e2.x));
    double det = ddot(e1, h);
    if (det > -EPS && det < EPS) return 0;
    d3 s = dsub(o, v0);
    double un = ddot(s, h);
    d3 q = D3(dcr(s.y, e1.z, s.z, e1.y), dcr(s.z, e1.x, s.x, e1.z), dcr(s.x, e1.y, s.y, e1.x));
    double vn = ddot(d, q);
    if (det > 0.0) {
        if (un < 0.0 || un > det || vn < 0.0 || un + vn > det) return 0;
    }
    else {
        if (un > 0.0 || un < det || vn > 0.0 || un + vn < det) return 0;
    }
    double t = ddot(e2, q) / det;
    if (t > EPS && t > t_min && t <= t_max) { /* t == t_max: exact tie, settled by the caller's tie rule */
        *t_out = t;
        return 1;
    }
    return 0;
}

static int obj_type(const orc_scene *s, int id)
{
    if (id < s->n_spheres) return 0;
    if (id < s->n_spheres + s->n_mspheres) return 1;
    return id < s->n_spheres + s->n_mspheres + s->n_triangles ? 2 : 3;
}

/* (base, rate) of v0 and the float edges e1(time), e2(time) of a moving triangle's pose (include/rrtb.h "rrtb_mtriangle") */
static void mtri_pose(const rrtb_mtriangle *m, float time, float base[3], float rate[3], float e1[3], float e2[3])
{
    float e1b[3], e1r[3], e2b[3], e2r[3];
    orc_mtriangle_record2(m, base, rate, e1b, e1r, e2b, e2r);
    for (int k = 0; k < 3; ++k) {
        e1[k] = e1r[k] == 0.0f ? e1b[k] : fmaf(e1r[k], time, e1b[k]);
        e2[k] = e2r[k] == 0.0f ? e2b[k] : fmaf(e2r[k], time, e2b[k]);
    }
}

static int hit_d(const orc_scene *s, int id, d3 o, d3 d, double time, double t_min, double t_max, double *t)
{
    int ty = obj_type(s, id);
    if (ty == 0) {
        const rrtb_sphere *sp = &s->spheres[id];
        return sphere_d(o, d, ldf(sp->center), (double)sp->radius, t_min, t_max, t);
    }
    if (ty == 1) {
        const rrtb_msphere *m = &s->mspheres[id - s->n_spheres];
        return sphere_d(o, d, msphere_center_d(m, time), (double)m->radius, t_min, t_max, t);
    }
    if (ty == 2) {
        const rrtb_triangle *tr = &s->triangles[id - s->n_spheres - s->n_mspheres];
        float e1[3], e2[3];
        for (int k = 0; k < 3; ++k) {
            e1[k] = tr->v1[k] - tr->v0[k];
            e2[k] = tr->v2[k] - tr->v0[k];
        }
        return triangle_d(o, d, ldf(tr->v0), e1, e2, t_min, t_max, t);
    }
    /* SURVEY 8f4: v0(time) = fma(rate, time, base) in double; the edges of the pose at `time` in float from the float
     * view of the time, as the float integrator evaluates them */
    float base[3], rate[3], e1[3], e2[3];
    mtri_pose(&s->mtriangles[id - s->n_spheres - s->n_mspheres - s->n_triangles], (float)time, base, rate, e1, e2);
    d3 v0 = D3(fma((double)rate[0], time, (double)base[0]), fma((double)rate[1], time, (double)base[1]),
               fma((double)rate[2], time, (double)base[2]));
    return triangle_d(o, d, v0, e1, e2, t_min, t_max, t);
}

static int wins_d(const orc_scene *s, double t, int id, double bt, int bid)
{
    if (bid < 0 || t < bt) return 1;
    if (t > bt) return 0;
    int ct = obj_type(s, id) >= 2, bt_tri = obj_type(s, bid) >= 2;
    if (ct != bt_tri) return !ct;
    return ct ? (id < bid) : (id > bid);
}

static d3 tri_normal_f(const rrtb_triangle *tr)
{
    float n[3];
    orc_triangle_normal(tr, n);
    return D3((double)n[0], (double)n[1], (double)n[2]);
}

/* rec7 = p(3), face-forwarded normal(3), front */
static void record_d(const orc_scene *s, int id, d3 o, d3 d, double time, double t, double *rec7, int *mat)
{
    d3 p = D3(fma(t, d.x, o.x), fma(t, d.y, o.y), fma(t, d.z, o.z));
    d3 n;
    int ty = obj_type(s, id);
    if (ty == 0) {
        const rrtb_sphere *sp = &s->spheres[id];
        double inv = 1.0 / (double)sp->radius;
        d3 c = ldf(sp->center);
        n = D3(inv * (p.x - c.x), inv * (p.y - c.y), inv * (p.z - c.z));
        *mat = sp->material;
    }
    else if (ty == 1) {
        const rrtb_msphere *m = &s->mspheres[id - s->n_spheres];
        double inv = 1.0 / (double)m->radius;
        d3 c = msphere_center_d(m, time);
        n = D3(inv * (p.x - c.x), inv * (p.y - c.y), inv * (p.z - c.z));
        *mat = m->material;
    }
    else if (ty == 2) {
        const rrtb_triangle *tr = &s->triangles[id - s->n_spheres - s->n_mspheres];
        n = tri_normal_f(tr);
        *mat = tr->material;
    }
    else { /* the float unit normal of the pose at the ray's time */
        const rrtb_mtriangle *m = &s->mtriangles[id - s->n_spheres - s->n_mspheres - s->n_triangles];
        float base[3], rate[3], e1[3], e2[3];
        mtri_pose(m, (float)time, base, rate, e1, e2);
        rrtb_triangle tr;
        for (int k = 0; k < 3; ++k) {
            tr.v0[k] = 0.0f;
            tr.v1[k] = e1[k]; /* v1 - v0 = e1 - 0 = e1 exactly */
            tr.v2[k] = e2[k];
        }
        n = tri_normal_f(&tr);
        *mat = m->material;
    }
    int front = (d.x * n.x + d.y * n.y) + d.z * n.z < 0.0;
    if (!front) n = D3(-n.x, -n.y, -n.z);
    std3(rec7, p);
    std3(rec7 + 3, n);
    rec7[6] = front ? 1.0 : 0.0;
}

static int box_hit_f(const float *bx, float pad, const float inv[3], const float ood[3], float t_min, float t_max)
{
    float lo = t_min, hi = t_max;
    for (int k = 0; k < 3; ++k) {
        float a = fmaf(bx[k] - pad, inv[k], ood[k]), b = fmaf(bx[3 + k] + pad, inv[k], ood[k]);
        lo = fmaxf(lo, fminf(a, b));
        hi = fminf(hi, fmaxf(a, b));
    }
    return lo <= hi;
}

/* closest hit; bvh may be NULL (flat scan).  The slab tests run in float on the float-rounded ray against the
 * padded boxes (conservative: the padding is 16x the rounding of the ray), the leaf tests in double. */
static int closest_d(const orc_scene *s, const orc_bvh *b, d3 o, d3 d, double time, double t_min, double *t_out)
{
    int n = orc_n_objects(s);
    double best = INFINITY;
    int bid = -1;
    if (!b || n < 2) {
        for (int id = 0; id < n; ++id) {
            double t;
            if (hit_d(s, id, o, d, time, t_min, best, &t) && wins_d(s, t, id, best, bid)) {
                best = t;
                bid = id;
            }
        }
        *t_out = best;
        return bid;
    }
    float df[3] = {(float)d.x, (float)d.y, (float)d.z}, of[3] = {(float)o.x, (float)o.y, (float)o.z}, inv[3], ood[3];
    for (int k = 0; k < 3; ++k) {
        float dk = fabsf(df[k]) < 1e-20f ? copysignf(1e-20f, df[k]) : df[k];
        inv[k] = 1.0f / dk;
        ood[k] = -of[k] * inv[k];
    }
    float tminf = nextafterf((float)t_min, 0.0f);
    int32_t stack[128];
    int sp = 0;
    stack[sp++] = 0;
    while (sp > 0) {
        int32_t node = stack[--sp];
        int32_t ch[2] = {b->left[node], b->right[node]};
        for (int c = 0; c < 2; ++c) {
            int32_t k = ch[c];
            const float *bx = k >= 0 ? b->node_box + 6 * (size_t)k : b->prim_box + 6 * (size_t)b->perm[~k];
            float tmaxf = isinf(best) ? INFINITY : nextafterf((float)best, INFINITY);
            if (!box_hit_f(bx, b->pad, inv, ood, tminf, tmaxf)) continue;
            if (k >= 0) {
                stack[sp++] = k;
            }
            else {
                int id = (int)b->perm[~k];
                double t;
                if (hit_d(s, id, o, d, time, t_min, best, &t) && wins_d(s, t, id, best, bid)) {
                    best = t;
                    bid = id;
                }
            }
        }
    }
    *t_out = best;
    return bid;
}

/* rays7: o d time (double).  rec7 optional. */
void orc_d_trace(const orc_scene *s, const orc_bvh *b, const double *rays7, int n, double t_min, int32_t *id, double *t,
                 double *rec7)
{
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; ++i) {
        const double *r = rays7 + 7 * (size_t)i;
        double tt;
        int bid = closest_d(s, b, ldd(r), ldd(r + 3), r[6], t_min, &tt);
        id[i] = bid;
        t[i] = bid >= 0 ? tt : -1.0;
        if (rec7) {
            double *o = rec7 + 7 * (size_t)i;
            memset(o, 0, 7 * sizeof(double));
            int mat;
            if (bid >= 0) record_d(s, bid, ldd(r), ldd(r + 3), r[6], tt, o, &mat);
        }
    }
}

static d3 unit_sphere_d(double x0, double x1)
{
    double z = fma(-2.0, x0, 1.0);
    double r = sqrt(fmax(0.0, fma(-z, z, 1.0)));
    double c, s;
    sincos2pi_d(x1, &c, &s);
    return D3(r * c, r * s, z);
}

/* material.h:21-32,48-57,76-109 in double; same Philox block layout as the float integrator */
static int scatter_d(const rrtb_material *m, d3 d_in, d3 n, int front, const uint32_t rnd[4], d3 *dir, d3 *att)
{
    if (m->type == RRTB_DIFFUSE_LIGHT) { /* never scatters; att = (double)Le */
        *dir = D3(0, 0, 0);
        *att = ldf(m->albedo);
        return 0;
    }
    if (m->type == RRTB_LAMBERTIAN) {
        d3 u = unit_sphere_d(u01d(rnd[0]), u01d(rnd[1]));
        d3 sd = D3(n.x + u.x, n.y + u.y, n.z + u.z);
        if (fabs(sd.x) < 1e-8 && fabs(sd.y) < 1e-8 && fabs(sd.z) < 1e-8) sd = n;
        *dir = sd;
        *att = ldf(m->albedo);
        return 1;
    }
    double inv = 1.0 / sqrt(ddot(d_in, d_in));
    d3 ud = D3(inv * d_in.x, inv * d_in.y, inv * d_in.z);
    double dn = ddot(ud, n);
    if (m->type == RRTB_METAL) {
        double k = -2.0 * dn;
        d3 r = D3(fma(k, n.x, ud.x), fma(k, n.y, ud.y), fma(k, n.z, ud.z));
        double fuzz = fabs(m->param < 1.0f ? (double)m->param : 1.0);
        if (fuzz > 0.0) {
            d3 u = unit_sphere_d(u01d(rnd[0]), u01d(rnd[1]));
            double ra = u01d(rnd[2]);
            double rb = (double)(rnd[3] >> 16) * 1.52587890625e-05, rc = (double)(rnd[3] & 0xFFFFu) * 1.52587890625e-05;
            double rad = fmax(ra, fmax(rb, rc)) * fuzz;
            r = D3(fma(rad, u.x, r.x), fma(rad, u.y, r.y), fma(rad, u.z, r.z));
        }
        *dir = r;
        *att = ldf(m->albedo);
        return ddot(r, n) > 0.0;
    }
    double ir = (double)m->param;
    double eta = front ? 1.0 / ir : ir;
    double cos_t = fmin(-dn, 1.0);
    double sin_t = sqrt(fmax(0.0, fma(-cos_t, cos_t, 1.0)));
    int cannot = eta * sin_t > 1.0;
    double r0 = (1.0 - eta) / (1.0 + eta);
    r0 = r0 * r0;
    double om = 1.0 - cos_t, om2 = om * om;
    double refl = fma(1.0 - r0, om2 * om2 * om, r0);
    if (cannot || refl > u01d(rnd[0])) {
        double k = -2.0 * dn;
        *dir = D3(fma(k, n.x, ud.x), fma(k, n.y, ud.y), fma(k, n.z, ud.z));
    }
    else {
        d3 p = D3(eta * fma(cos_t, n.x, ud.x), eta * fma(cos_t, n.y, ud.y), eta * fma(cos_t, n.z, ud.z));
        double k = -sqrt(fabs(1.0 - ddot(p, p)));
        *dir = D3(fma(k, n.x, p.x), fma(k, n.y, p.y), fma(k, n.z, p.z));
    }
    *att = D3(1, 1, 1);
    return 1;
}

/* in16 per item (double): ray o(3) d(3) time, p(3), n(3), front, material, unused; out8: dir(3) att(3) ok - */
void orc_d_scatter(const orc_scene *s, const double *in16, const uint32_t *rnd4, int n, double *out8)
{
    for (int i = 0; i < n; ++i) {
        const double *in = in16 + 16 * (size_t)i;
        double *o = out8 + 8 * (size_t)i;
        d3 dir, att;
        int ok = scatter_d(&s->materials[(int)in[14]], ldd(in + 3), ldd(in + 10), in[13] != 0.0, rnd4 + 4 * (size_t)i, &dir, &att);
        std3(o, dir);
        std3(o + 3, att);
        o[6] = ok ? 1.0 : 0.0;
        o[7] = 0.0;
    }
}

/* bg: the constant background that replaces the sky, or NULL for the sky */
static void path_d(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int pixel, int sample, int max_depth,
                   uint64_t seed, double *rgb, orc_counters *cnt)
{
    double ray7[7];
    orc_d_camera_ray(&s->cam, W, H, pixel, sample, seed, ray7);
    d3 o = ldd(ray7), d = ldd(ray7 + 3);
    double time = ray7[6];
    d3 thr = D3(1, 1, 1);
    rgb[0] = rgb[1] = rgb[2] = 0.0;
    cnt->paths++;
    for (int b = 0; b < max_depth; ++b) {
        double t;
        int id = closest_d(s, bvh, o, d, time, 0.001, &t);
        cnt->rays++;
        if (id < 0 && bg) {
            rgb[0] = thr.x * (double)bg[0];
            rgb[1] = thr.y * (double)bg[1];
            rgb[2] = thr.z * (double)bg[2];
            return;
        }
        if (id < 0) {
            double uy = d.y * (1.0 / sqrt(ddot(d, d)));
            double tt = 0.5 * (uy + 1.0);
            rgb[0] = thr.x * fma(tt, 0.5, 1.0 - tt);
            rgb[1] = thr.y * fma(tt, 0.7, 1.0 - tt);
            rgb[2] = thr.z * fma(tt, 1.0, 1.0 - tt);
            return;
        }
        cnt->hits++;
        double rec[7];
        int mat;
        record_d(s, id, o, d, time, t, rec, &mat);
        uint32_t rnd[4];
        rng_block(seed, (uint32_t)pixel, (uint32_t)sample, 2u + (uint32_t)b, rnd);
        d3 dir, att;
        if (!scatter_d(&s->materials[mat], d, ldd(rec + 3), rec[6] != 0.0, rnd, &dir, &att)) {
            if (s->materials[mat].type == RRTB_DIFFUSE_LIGHT) { /* emitter: throughput x Le (att = (double)Le) */
                rgb[0] = thr.x * att.x;
                rgb[1] = thr.y * att.y;
                rgb[2] = thr.z * att.z;
            }
            return; /* else absorbed: black */
        }
        thr = D3(thr.x * att.x, thr.y * att.y, thr.z * att.z);
        o = ldd(rec);
        d = dir;
    }
}

static inline uint64_t to_fixed_d(double x, double clamp)
{
    if (!(x > 0.0)) return 0;
    if (x > clamp) x = clamp;
    return (uint64_t)llrint(x * 1099511627776.0);
}

/* out_rgb: 3*W*H double sums (bottom-up); out_fixed optional */
void orc_d_render(const orc_scene *s, const orc_bvh *bvh, int W, int H, int spp, int max_depth, uint64_t seed, double *out_rgb,
                  uint64_t *out_fixed, orc_counters *cnt)
{
    orc_d_render_bg(s, NULL, bvh, W, H, spp, max_depth, seed, out_rgb, out_fixed, cnt);
}

void orc_d_render_bg(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                     uint64_t seed, double *out_rgb, uint64_t *out_fixed, orc_counters *cnt)
{
    orc_counters total;
    memset(&total, 0, sizeof(total));
    const double clamp = orc_fixed_clamp(spp);
#pragma omp parallel
    {
        orc_counters local;
        memset(&local, 0, sizeof(local));
#pragma omp for schedule(dynamic, 4)
        for (int j = 0; j < H; ++j)
            for (int i = 0; i < W; ++i) {
                int pixel = j * W + i;
                uint64_t acc[3] = {0, 0, 0};
                for (int sm = 0; sm < spp; ++sm) {
                    double rgb[3];
                    path_d(s, bg, bvh, W, H, pixel, sm, max_depth, seed, rgb, &local);
                    for (int k = 0; k < 3; ++k) acc[k] += to_fixed_d(rgb[k], clamp);
                }
                for (int k = 0; k < 3; ++k) {
                    if (out_fixed) out_fixed[3 * (size_t)pixel + k] = acc[k];
                    if (out_rgb) out_rgb[3 * (size_t)pixel + k] = (double)acc[k] * 9.094947017729282e-13;
                }
            }
#pragma omp critical
        {
            total.rays += local.rays;
            total.hits += local.hits;
            total.paths += local.paths;
        }
    }
    if (cnt) *cnt = total;
}
