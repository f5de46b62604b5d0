/* lights_f64.c -- TEST INFRASTRUCTURE ONLY: the double oracle with lights (lights.h).  The oracle source is compiled
 * into this translation unit, so the static helpers below are exactly the ones orc_d_render uses; the emitted and
 * background terms are one double product per channel, as __dmul_rn(throughput, (double)L) in PathF64::const_fixed. */
#include "../../oracle/rrt_oracle_f64.c"
#include "lights.h"

static int scatter_d_lit(const rrtb_material *m, d3 d_in, d3 n, int front, const uint32_t rnd[4], d3 *dir, d3 *att)
{
    if (m->type == RRTB_DIFFUSE_LIGHT) {
        *dir = D3(0, 0, 0);
        *att = ldf(m->albedo);
        return 0;
    }
    return scatter_d(m, d_in, n, front, rnd, dir, att);
}

void orc_l_d_scatter(const orc_scene *s, const double *in16, const uint32_t *rnd4, int n, double *out8)
{
    for (int i = 0; i < n; ++i) {
        const double *in = in16 + 16 * (size_t)i;
        double *o = out8 + 8 * (size_t)i;
        d3 dir, att;
        int ok = scatter_d_lit(&s->materials[(int)in[14]], ldd(in + 3), ldd(in + 10), in[13] != 0.0, rnd4 + 4 * (size_t)i,
                               &dir, &att);
        std3(o, dir);
        std3(o + 3, att);
        o[6] = ok ? 1.0 : 0.0;
        o[7] = 0.0;
    }
}

/* path_d with the emitted and background terms */
static void path_d_lit(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int pixel, int sample,
                       int max_depth, uint64_t seed, double *rgb, orc_counters *cnt)
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
        if (id < 0 && bg) { /* background x throughput */
            rgb[0] = thr.x * (double)bg[0];
            rgb[1] = thr.y * (double)bg[1];
            rgb[2] = thr.z * (double)bg[2];
            return;
        }
        if (id < 0) { /* the sky, as path_d */
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
        if (!scatter_d_lit(&s->materials[mat], d, ldd(rec + 3), rec[6] != 0.0, rnd, &dir, &att)) {
            if (s->materials[mat].type == RRTB_DIFFUSE_LIGHT) { /* emitter: throughput x Le (att = (double)Le) */
                rgb[0] = thr.x * att.x;
                rgb[1] = thr.y * att.y;
                rgb[2] = thr.z * att.z;
            }
            return;
        }
        thr = D3(thr.x * att.x, thr.y * att.y, thr.z * att.z);
        o = ldd(rec);
        d = dir;
    }
}

void orc_l_d_render(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
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
                    path_d_lit(s, bg, bvh, W, H, pixel, sm, max_depth, seed, rgb, &local);
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
