/* rrt_oracle.h -- TEST INFRASTRUCTURE ONLY: the CPU oracle for the rrt path-tracing hot path.
 *
 * A plain-C restatement of (a) the reference's estimator / intersection / material semantics and
 * (b) the canonical LBVH + Philox algorithms the CUDA product implements (SURVEY Appendix B, D).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this library.
 * It is never linked into, imported by or called from the product (rrt_b200/, librrtb200.so).
 *
 * Parity status: PINNED by execution of the reference itself -- the reference has no golden
 * vectors or tests of its own (SURVEY 4, 8c), so this oracle is checked against
 * oracle/_ref/libref_{f,d}.so (the unmodified reference headers compiled by oracle/Makefile) in
 * tests/test_oracle_vs_reference.py and against fixtures generated from that harness
 * (tests/golden/, tools/make_golden.py).
 *
 * The scene structs are the public C ABI ones (include/rrtb.h) so the same arrays feed both sides.
 *
 * Lights (DESIGN f5) have no reference counterpart and are parity-unpinned: a RRTB_DIFFUSE_LIGHT material never
 * scatters and ends the path with throughput x Le (Le = its albedo), and the background of orc_render_bg /
 * orc_d_render_bg, when not NULL, replaces the sky with throughput x background.  Both terms are float products in the
 * float integrator and one double product of the float-to-double value per channel in the double one, in the order of
 * the product's PathF32 / PathF64 ::const_fixed.  A scene without a RRTB_DIFFUSE_LIGHT material, rendered with the
 * sky, reaches neither term, so on it every entry point is exactly the parity-pinned estimator above.
 */
#ifndef RRT_ORACLE_H
#define RRT_ORACLE_H

#include "../include/rrtb.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct orc_scene {
    rrtb_camera cam;
    const rrtb_material *materials; int n_materials;
    const rrtb_sphere *spheres;     int n_spheres;
    const rrtb_msphere *mspheres;   int n_mspheres;
    const rrtb_triangle *triangles; int n_triangles;
    const rrtb_mtriangle *mtriangles; int n_mtriangles; /* SURVEY 8f4: translating instance triangles (ids after triangles) */
} orc_scene;

typedef struct orc_bvh {
    int n;              /* primitives */
    uint32_t *morton;   /* [n]   object-id order */
    uint32_t *perm;     /* [n]   sorted position -> object id */
    int32_t *left;      /* [n-1] >=0 internal, <0 leaf ~k */
    int32_t *right;     /* [n-1] */
    int32_t *parent;    /* [2n-1] */
    float *node_box;    /* [6(n-1)] */
    float *prim_box;    /* [6n]  object-id order */
    float pad;          /* absolute padding applied to boxes during traversal */
} orc_bvh;

typedef struct orc_counters { /* per-ray work counters (SURVEY 8d: V_box, V_sph, V_msph, V_tri, h) */
    uint64_t rays, box_tests, sphere_tests, msphere_tests, triangle_tests, hits, paths;
} orc_counters;

/* Philox4x32-10 (Salmon et al., SC 2011). */
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* (x >> 8) * 2^-24, in [0,1) */
float orc_u01(uint32_t x);
/* (cos, sin) of 2*pi*(u - 0.5), the deterministic polynomial both sides use for sampling */
void orc_sincos2pi(float u, float *c, float *s);

/* camera.h:8-29 */
void orc_camera_derive(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov,
                       float aspect, float aperture, float focus, float t0, float t1, rrtb_camera *out);
/* rrt.cu:112-114 + camera.h:31-38 with the Philox streams of the product. ray7 = o d time */
void orc_camera_ray(const rrtb_camera *cam, int W, int H, int pixel, int sample, uint64_t seed, float *ray7);

/* per-primitive tests with the product's precision policy. id = object id. returns 0/1.
 * rec7 (optional) = p(3), face-forwarded normal(3), front_face */
int orc_hit_object(const orc_scene *s, int id, const float *ray7, float t_min, float t_max, float *t, float *rec7);
/* hittable_list.h:95-117 semantics: flat scan, object-id order, shrinking t_max */
void orc_trace_scan(const orc_scene *s, const float *rays7, int n, float t_min, int32_t *id, float *t, float *rec7);

/* canonical LBVH (SURVEY Appendix D) */
orc_bvh *orc_bvh_build(const orc_scene *s);
void orc_bvh_free(orc_bvh *b);
void orc_trace_bvh(const orc_scene *s, const orc_bvh *b, const float *rays7, int n, float t_min, int32_t *id,
                   float *t, float *rec7, orc_counters *cnt);

/* the traversal tree of the product (rrt_oracle_wide.c): the SAH rebuild of the LBVH's lower subtrees, the refit of
 * the Morton top, the 4-wide collapse and its node encoding, restated in float in the GPU's operation order */
typedef struct orc_wide_counters {
    int32_t sort_small;        /* 1: one-block bitonic sort (n <= 2048), 0: radix sort */
    int32_t rebuild_shape;     /* k_sah_rebuild<1024> (n <= 4096) or <256>; 0: no rebuild (n < 3) */
    int32_t n_roots;           /* rebuilt subtrees */
    int32_t block_splits;      /* binned splits of runs of more than 128 by the whole block (shape 1024 only) */
    int32_t block_median_coincident, block_median_budget; /* ... of them median splits: no plane / depth budget */
    int32_t warp_splits;       /* binned splits by one warp (runs of 5 or more) */
    int32_t warp_median_coincident, warp_median_budget;
    int32_t small_splits;      /* exact splits of runs of 2..4 boxes */
    int32_t small_halved;      /* ... of them halved: no finite cost or depth budget */
    int32_t refit_parent;      /* leaves directly under a node of more than 512 leaves (k_refit_upper parent rule) */
    int32_t refit_grandparent; /* leaves of a 2-leaf node under a node of more than 512 leaves (grandparent rule) */
    int32_t max_binary_depth;  /* deepest leaf of the binary traversal tree, root = 0 */
    int32_t max_wide_depth;    /* deepest 4-wide node, root = 0 */
    float pad;                 /* the traversal-box padding the nodes were encoded with: 2^-20 max(largest |coordinate| of
                                * a primitive box, max_k |origin_k| + lens radius), computed here (tests compare it with
                                * orc_bvh.pad) */
} orc_wide_counters;

typedef struct orc_wide {
    int32_t n_nodes, words_per_node; /* 24 words per node, 40 per motion node (rrtb_device.cuh) */
    uint32_t *words;                 /* [n_nodes * words_per_node], canonical order: pre-order, children in slot order */
    int32_t n_tasks, n_items;
    int32_t *tasks; /* [n_tasks * 7] per split: path (0 block, 1 warp, 2 exact), first item, count, choice (axis * 32 + bin,
                     * the left mask of an exact split, -1 for a binned median split), how (0 SAH, 1 no plane / no
                     * finite cost, 2 depth budget), level below the subtree root, budget (63 - canonical depth of the
                     * subtree root) */
    int32_t *items;     /* the sorted positions of each split's run, in run order */
    float *prim_box01;  /* [12 n] object-id order: lo, hi at camera time0, lo, hi at camera time1 (k_prepare) */
    int32_t *left2, *right2; /* [max(n - 1, 1)] the binary traversal tree the collapse reads (rebuilt subtrees and the
                              * Morton top; the canonical LBVH for n < 3): >= 0 node, < 0 leaf ~sorted position */
    float *node_box2;        /* [6 max(n - 1, 1)] its node boxes, min xyz, max xyz */
    orc_wide_counters cnt;
} orc_wide;

/* motion: 40-word motion nodes with both ends of the shutter (the caller applies the library's rule) */
orc_wide *orc_wide_build(const orc_scene *s, int motion);
void orc_wide_free(orc_wide *w);
/* float -> IEEE half rounded toward +inf, bits (the half extents of the traversal nodes) */
uint16_t orc_f16_up(float h);

/* material.h scatter with an explicit Philox block. in16/out8 as rrtb_scatter.  An emitter reports direction 0,
 * attenuation Le, not scattered. */
void orc_scatter(const orc_scene *s, const float *in16, const uint32_t *rnd4, int n, float *out8);

/* per-sample radiance clamp of a render of spp samples in all: min(2^20, 2^(23 - ceil(log2 spp))), so that a pixel's
 * sum of spp fixed-point samples stays <= 2^63 (the product's fixed_clamp, rrt_b200/csrc/rrtb_device.cuh) */
static inline float orc_fixed_clamp(int spp)
{
    int lg = 0;
    while (lg < 31 && (1u << lg) < (unsigned)spp) ++lg;
    int e = 23 - lg;
    return (float)(1u << (e > 20 ? 20 : (e < 0 ? 0 : e)));
}

/* the estimator (rrt.cu:42-79,109-121 semantics, product RNG). out_rgb = 3*W*H float sums, bottom-up.
 * bvh may be NULL (flat scan). Pixels with (tile_index % world) != rank are left 0 when world > 1.
 * Each sample's radiance is clamped to orc_fixed_clamp(spp) (spp = the whole render's, also for a shard). */
void orc_render(const orc_scene *s, const orc_bvh *bvh, int W, int H, int spp, int max_depth, uint64_t seed,
                int rank, int world, int shard_mode, float *out_rgb, uint64_t *out_fixed, orc_counters *cnt);
/* orc_render under a constant background: background[3] replaces the sky; NULL is the sky (orc_render) */
void orc_render_bg(const orc_scene *s, const float *background, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                   uint64_t seed, int rank, int world, int shard_mode, float *out_rgb, uint64_t *out_fixed,
                   orc_counters *cnt);
/* ray_color for an explicit primary ray ((pixel, sample) only key the bounce RNG) */
void orc_radiance(const orc_scene *s, const orc_bvh *bvh, const float *ray7, int pixel, int sample, int max_depth,
                  uint64_t seed, float *rgb, orc_counters *cnt);
/* one camera path; returns radiance in rgb[3] */
void orc_path(const orc_scene *s, const orc_bvh *bvh, int W, int H, int pixel, int sample, int max_depth,
              uint64_t seed, float *rgb, orc_counters *cnt);

/* triangle.h:9-15: the float unit face normal the product stores in its leaf record */
void orc_triangle_normal(const rrtb_triangle *tr, float n[3]);
/* a moving triangle as the product's leaf record defines it (include/rrtb.h "rrtb_mtriangle"):
 * rate[k] = delta[k] / (time1 - time0), base[k] = fma(-rate[k], time0, v0[k]); v0(time) = fma(rate, time, base) */
void orc_mtriangle_record(const rrtb_mtriangle *m, float base[3], float rate[3], float e1[3], float e2[3]);
/* the full record: (base, rate) of v0, of e1 = v1 - v0 and of e2 = v2 - v0 (extra1 / extra2 make the edges move) */
void orc_mtriangle_record2(const rrtb_mtriangle *m, float base[3], float rate[3], float e1b[3], float e1r[3], float e2b[3], float e2r[3]);
static inline int orc_n_objects(const orc_scene *s) { return s->n_spheres + s->n_mspheres + s->n_triangles + s->n_mtriangles; }

/* ---- the DOUBLE integrator (rrt_oracle_f64.c; SURVEY 8f1): FP_T = double semantics over the same float scene ---- */
void orc_d_camera_ray(const rrtb_camera *cam, int W, int H, int pixel, int sample, uint64_t seed, double *ray7);
/* closest hit, leaf tests in double; b may be NULL (flat scan). rec7 optional = p(3) n(3) front */
void orc_d_trace(const orc_scene *s, const orc_bvh *b, const double *rays7, int n, double t_min, int32_t *id, double *t,
                 double *rec7);
void orc_d_scatter(const orc_scene *s, const double *in16, const uint32_t *rnd4, int n, double *out8);
void orc_d_render(const orc_scene *s, const orc_bvh *bvh, int W, int H, int spp, int max_depth, uint64_t seed, double *out_rgb,
                  uint64_t *out_fixed, orc_counters *cnt);
/* orc_d_render under a constant background, as orc_render_bg */
void orc_d_render_bg(const orc_scene *s, const float *background, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                     uint64_t seed, double *out_rgb, uint64_t *out_fixed, orc_counters *cnt);

/* color.h:8-23 */
void orc_tonemap_rgb8(const float *rgb_sum, int W, int H, int spp, uint8_t *rgb8_topdown);

#ifdef __cplusplus
}
#endif
#endif
