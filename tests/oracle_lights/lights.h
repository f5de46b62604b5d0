/* lights.h -- TEST INFRASTRUCTURE ONLY: diffuse_light emitters and a constant background for the CPU oracle.
 *
 * The product's lights (include/rrtb.h RRTB_DIFFUSE_LIGHT, rrtb_scene_stage_background) have no reference counterpart.
 * These entry points restate them over the unchanged oracle: lights_f32.c and lights_f64.c each compile one oracle
 * source (oracle/rrt_oracle.c, oracle/rrt_oracle_f64.c) into the same translation unit and reuse its intersection,
 * LBVH, camera, Philox and material code; only the estimator loop is new.  Semantics (both integrators):
 *   - a segment that hits a RRTB_DIFFUSE_LIGHT material ends the path with throughput x Le (Le = the albedo): float
 *     products in the float integrator, double products of the float-to-double Le in the double one, in the order of
 *     the product's PathF32 / PathF64 ::const_fixed
 *   - with bg != NULL a segment that leaves the scene adds throughput x bg instead of the sky; bg == NULL is the sky
 *   - every sample is clamped to orc_fixed_clamp(spp) like any other
 * The scatter hooks report an emitter as not scattered: direction 0, attenuation Le, scattered 0.
 * With no emitter and bg == NULL every function returns exactly what its oracle counterpart returns. */
#ifndef RRTB_ORACLE_LIGHTS_H
#define RRTB_ORACLE_LIGHTS_H
#include "../../oracle/rrt_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* orc_render / orc_scatter with lights */
void orc_l_render(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                  uint64_t seed, int rank, int world, int shard_mode, float *out_rgb, uint64_t *out_fixed,
                  orc_counters *cnt);
void orc_l_scatter(const orc_scene *s, const float *in16, const uint32_t *rnd4, int n, float *out8);
/* orc_d_render / orc_d_scatter with lights */
void orc_l_d_render(const orc_scene *s, const float *bg, const orc_bvh *bvh, int W, int H, int spp, int max_depth,
                    uint64_t seed, double *out_rgb, uint64_t *out_fixed, orc_counters *cnt);
void orc_l_d_scatter(const orc_scene *s, const double *in16, const uint32_t *rnd4, int n, double *out8);

#ifdef __cplusplus
}
#endif
#endif
