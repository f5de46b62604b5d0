/* lights_f32.c -- TEST INFRASTRUCTURE ONLY: the float oracle with lights (lights.h).  The oracle source is compiled
 * into this translation unit, so the static helpers below are exactly the ones orc_render uses. */
#include "../../oracle/rrt_oracle.c"
#include "lights.h"

/* scatter_one, except that an emitter never scatters (book 2 diffuse_light) */
static int scatter_lit(const rrtb_material *m, f3 d_in, f3 n, int front, const uint32_t rnd[4], f3 *dir, f3 *att)
{
    if (m->type == RRTB_DIFFUSE_LIGHT) {
        *dir = F3(0.0f, 0.0f, 0.0f);
        *att = ld3(m->albedo);
        return 0;
    }
    return scatter_one(m, d_in, n, front, rnd, dir, att);
}

void orc_l_scatter(const orc_scene *s, const float *in16, const uint32_t *rnd4, int n, float *out8)
{
    for (int i = 0; i < n; ++i) {
        const float *in = in16 + 16 * (size_t)i;
        float *o = out8 + 8 * (size_t)i;
        f3 dir, att;
        int ok = scatter_lit(&s->materials[(int)in[14]], ld3(in + 3), ld3(in + 10), in[13] != 0.0f, rnd4 + 4 * (size_t)i,
                             &dir, &att);
        st3(o, dir);
        st3(o + 3, att);
        o[6] = ok ? 1.0f : 0.0f;
        o[7] = 0.0f;
    }
}

/* orc_radiance with the emitted and background terms */
static void radiance_lit(const orc_scene *s, const float *bg, const orc_bvh *bvh, const float *ray7, int pixel, int sample,
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
        if (id < 0 && bg) { /* background x throughput */
            rgb[0] = thr.x * bg[0];
            rgb[1] = thr.y * bg[1];
            rgb[2] = thr.z * bg[2];
            return;
        }
        if (id < 0) { /* sky, rrt.cu:68-75 (as orc_radiance) */
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
        if (!scatter_lit(&s->materials[mat], d, ld3(rec + 3), rec[6] != 0.0f, rnd, &dir, &att)) {
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
}

void orc_l_render(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                  uint64_t seed, int rank, int world, int shard_mode, float *out_rgb, uint64_t *out_fixed,
                  orc_counters *cnt)
{
    orc_counters total;
    memset(&total, 0, sizeof(total));
    int tiles_x = (W + 7) / 8;
    const float clamp = orc_fixed_clamp(spp);
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
                if (world > 1 && shard_mode == RRTB_SHARD_TILES) mine = ((j / 4) * tiles_x + (i / 8)) % world == rank;
                if (mine) {
                    for (int sm = 0; sm < spp; ++sm) {
                        if (world > 1 && shard_mode == RRTB_SHARD_SAMPLES && (sm % world) != rank) continue;
                        float ray7[7], rgb[3];
                        orc_camera_ray(&s->cam, W, H, pixel, sm, seed, ray7);
                        radiance_lit(s, bg, bvh, ray7, pixel, sm, max_depth, seed, rgb, &local);
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
