/* aov_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU checker of the first-hit AOVs (include/rrtb.h rrtb_render_aov).
 *
 * Built on the oracle's public entry points alone (oracle/rrt_oracle.h): its camera rays (orc_camera_ray,
 * orc_d_camera_ray) and its closest-hit queries with their hit records (orc_trace_bvh / orc_trace_scan, orc_d_trace).
 * tests/test_aov.py compiles it at test time against oracle/liboracle.so; nothing under rrt_b200/ uses it.
 *
 * Per pixel and sample 0 .. spp-1 the camera ray and one closest-hit query (t_min 0.001); on a hit the clamped albedo,
 * the face-forwarded normal and t |d| are added, widened, to double sums in sample order (a miss adds nothing), and each
 * mean is one double division rounded once to float: the GPU's order.  The pixels of tiles with (tile % world) != rank
 * are 0.  albedo3 / normal3 = 3*W*H floats, depth / coverage = W*H, bottom-up.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "rrt_oracle.h"

typedef struct aov_sums { /* one pixel's sums in sample order */
    double al[3], nm[3], dist;
    int n_hit;
} aov_sums;

/* the material of object `id` (object-id order: spheres, moving spheres, triangles, moving triangles) */
static const rrtb_material *material_of(const orc_scene *s, int id)
{
    if (id < s->n_spheres) return &s->materials[s->spheres[id].material];
    id -= s->n_spheres;
    if (id < s->n_mspheres) return &s->materials[s->mspheres[id].material];
    id -= s->n_mspheres;
    if (id < s->n_triangles) return &s->materials[s->triangles[id].material];
    return &s->materials[s->mtriangles[id - s->n_triangles].material];
}

/* the material's attenuation clamped per channel to [0, 1]: dielectric 1, else the albedo (an emitter's Le) */
static void aov_albedo(const rrtb_material *m, float al[3])
{
    for (int k = 0; k < 3; ++k) al[k] = m->type == RRTB_DIELECTRIC ? 1.0f : fminf(fmaxf(m->albedo[k], 0.0f), 1.0f);
}

/* the pixels rank `rank` of `world` owns (interleaved 8x4-pixel tiles), in row order; returns their count */
static int owned_pixels(int W, int H, int rank, int world, int *pix)
{
    int n = 0;
    for (int j = 0; j < H; ++j)
        for (int i = 0; i < W; ++i)
            if (world <= 1 || ((j / 4) * ((W + 7) / 8) + i / 8) % world == rank) pix[n++] = j * W + i;
    return n;
}

static void store(const aov_sums *a, int spp, int pixel, float *albedo3, float *normal3, float *depth, float *coverage)
{
    for (int k = 0; k < 3; ++k) {
        albedo3[3 * (size_t)pixel + k] = (float)(a->al[k] / (double)spp);
        normal3[3 * (size_t)pixel + k] = (float)(a->nm[k] / (double)spp);
    }
    depth[pixel] = a->n_hit ? (float)(a->dist / (double)a->n_hit) : 0.0f;
    coverage[pixel] = (float)((double)a->n_hit / (double)spp);
}

/* the float integrator; bvh NULL: the flat scan */
void aov_render(const orc_scene *s, const orc_bvh *bvh, int W, int H, int spp, uint64_t seed, int rank, int world,
                float *albedo3, float *normal3, float *depth, float *coverage)
{
    const size_t np = (size_t)W * H;
    memset(albedo3, 0, 3 * np * sizeof(float));
    memset(normal3, 0, 3 * np * sizeof(float));
    memset(depth, 0, np * sizeof(float));
    memset(coverage, 0, np * sizeof(float));
    int *pix = malloc(np * sizeof(int));
    const int n = owned_pixels(W, H, rank, world, pix);
    aov_sums *sums = calloc((size_t)n > 0 ? (size_t)n : 1, sizeof(aov_sums));
    float *rays = malloc(7 * (size_t)n * sizeof(float) + 1), *t = malloc((size_t)n * sizeof(float) + 1);
    float *rec = malloc(7 * (size_t)n * sizeof(float) + 1);
    int32_t *id = malloc((size_t)n * sizeof(int32_t) + 1);
    for (int sm = 0; sm < spp; ++sm) {
        for (int k = 0; k < n; ++k) orc_camera_ray(&s->cam, W, H, pix[k], sm, seed, rays + 7 * (size_t)k);
        if (bvh) orc_trace_bvh(s, bvh, rays, n, 0.001f, id, t, rec, NULL);
        else orc_trace_scan(s, rays, n, 0.001f, id, t, rec);
        for (int k = 0; k < n; ++k) {
            if (id[k] < 0) continue;
            const float *d = rays + 7 * (size_t)k + 3, *r = rec + 7 * (size_t)k;
            float al[3];
            aov_albedo(material_of(s, id[k]), al);
            aov_sums *a = &sums[k];
            for (int c = 0; c < 3; ++c) {
                a->al[c] += (double)al[c];
                a->nm[c] += (double)r[3 + c];
            }
            a->dist += (double)(t[k] * sqrtf(fmaf(d[2], d[2], fmaf(d[1], d[1], d[0] * d[0])))); /* t |d| */
            ++a->n_hit;
        }
    }
    for (int k = 0; k < n; ++k) store(&sums[k], spp, pix[k], albedo3, normal3, depth, coverage);
    free(pix); free(sums); free(rays); free(t); free(rec); free(id);
}

/* the double integrator: ray, normal and distance in double; bvh NULL: the flat scan */
void aov_d_render(const orc_scene *s, const orc_bvh *bvh, int W, int H, int spp, uint64_t seed, int rank, int world,
                  float *albedo3, float *normal3, float *depth, float *coverage)
{
    const size_t np = (size_t)W * H;
    memset(albedo3, 0, 3 * np * sizeof(float));
    memset(normal3, 0, 3 * np * sizeof(float));
    memset(depth, 0, np * sizeof(float));
    memset(coverage, 0, np * sizeof(float));
    int *pix = malloc(np * sizeof(int));
    const int n = owned_pixels(W, H, rank, world, pix);
    aov_sums *sums = calloc((size_t)n > 0 ? (size_t)n : 1, sizeof(aov_sums));
    double *rays = malloc(7 * (size_t)n * sizeof(double) + 1), *t = malloc((size_t)n * sizeof(double) + 1);
    double *rec = malloc(7 * (size_t)n * sizeof(double) + 1);
    int32_t *id = malloc((size_t)n * sizeof(int32_t) + 1);
    for (int sm = 0; sm < spp; ++sm) {
        for (int k = 0; k < n; ++k) orc_d_camera_ray(&s->cam, W, H, pix[k], sm, seed, rays + 7 * (size_t)k);
        orc_d_trace(s, bvh, rays, n, 0.001, id, t, rec);
        for (int k = 0; k < n; ++k) {
            if (id[k] < 0) continue;
            const double *d = rays + 7 * (size_t)k + 3, *r = rec + 7 * (size_t)k;
            float al[3];
            aov_albedo(material_of(s, id[k]), al);
            aov_sums *a = &sums[k];
            for (int c = 0; c < 3; ++c) {
                a->al[c] += (double)al[c];
                a->nm[c] += r[3 + c];
            }
            a->dist += t[k] * sqrt(fma(d[2], d[2], fma(d[1], d[1], d[0] * d[0]))); /* t |d| */
            ++a->n_hit;
        }
    }
    for (int k = 0; k < n; ++k) store(&sums[k], spp, pix[k], albedo3, normal3, depth, coverage);
    free(pix); free(sums); free(rays); free(t); free(rec); free(id);
}
