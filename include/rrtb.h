/* rrtb.h -- C ABI of librrtb200.so: the B200-native path-tracing core behind rrt's renderer seam.
 *
 * This is the drop-in boundary for ONE path of rogerallen/rrt: the renderer that sits behind
 * `class Rrt` (reference rrt.h:14-48; implementations rrt.cu / rrt.cpp chosen at link time,
 * reference Makefile:21-22).  Every entry point below names the reference interface it replaces
 * (file:line under /root/reference).  Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions
 *   - every function returns 0 on success, a negative rrtb_status on failure; the library never
 *     calls exit() (the reference does: rrt.cu:31-40) -- the `Rrt` shim in rrt_b200/host maps a
 *     failure back to the reference's message + exit(99).
 *   - one context = one GPU.  Multi-GPU = one context (normally one process) per GPU, each
 *     rendering the shard (rank, world) of the same image; the shards are disjoint-or-additive in a
 *     64-bit fixed-point accumulator, so any reduction order gives bit-identical images.
 *   - there is NO CPU fallback: without a CUDA device rrtb_create fails with RRTB_ERR_NO_DEVICE.
 *   - framebuffer layout is the reference's: index j*W+i, j = 0 is the BOTTOM scanline, value =
 *     SUM (not mean) over samples of per-sample radiance (rrt.cu:109-121).
 */
#ifndef RRTB_H
#define RRTB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RRTB_ABI_VERSION 3

typedef enum rrtb_status {
    RRTB_OK = 0,
    RRTB_ERR_INVALID = -1,   /* bad argument */
    RRTB_ERR_NO_DEVICE = -2, /* no CUDA device / device index out of range */
    RRTB_ERR_CUDA = -3,      /* a CUDA call failed; see rrtb_last_error */
    RRTB_ERR_NO_SCENE = -4,  /* render/trace before rrtb_scene_set */
    RRTB_ERR_IO = -5,        /* file could not be opened (reference exit code 2, scene.h:220-223) */
    RRTB_ERR_PARSE = -6,     /* malformed scene (reference exit codes 1/3/4) */
    RRTB_ERR_NOMEM = -7
} rrtb_status;

/* ---- scene vocabulary (reference scene.h:43-54,183-208; camera.h:40-48) ------------------------
 * All float, exactly the values the reference's float build (`rrt`) would hold. */

/* RRTB_DIFFUSE_LIGHT (book 2's diffuse_light; the reference has no lights): an emitter.  It emits its albedo as the
 * radiance Le on both faces and never scatters: a segment that hits it ends the path and adds throughput x Le to the
 * pixel, clamped by the same per-sample clamp C as the sky (rrtb_render_params.spp), so emitted radiance above C is
 * clipped (at spp = 2^23, C = 1).  Le is not validated, as albedos are not; a negative component adds 0. */
enum { RRTB_LAMBERTIAN = 0, RRTB_METAL = 1, RRTB_DIELECTRIC = 2, RRTB_DIFFUSE_LIGHT = 3 }; /* scene.h:183 */

typedef struct rrtb_camera { /* the derived fields of camera.h:8-29 */
    float origin[3];
    float lower_left_corner[3];
    float horizontal[3];
    float vertical[3];
    float u[3], v[3], w[3];
    float lens_radius;
    float time0, time1; /* shutter open/close */
} rrtb_camera;

typedef struct rrtb_material {
    int32_t type;    /* RRTB_LAMBERTIAN | RRTB_METAL | RRTB_DIELECTRIC | RRTB_DIFFUSE_LIGHT */
    float albedo[3]; /* lambertian, metal; diffuse_light: emitted radiance Le */
    float param;     /* metal: fuzz (clamped to <= 1 at use, material.h:48); dielectric: index of refraction */
} rrtb_material;

typedef struct rrtb_sphere { /* sphere.h:28-31 */
    float center[3];
    float radius;
    int32_t material;
} rrtb_sphere;

typedef struct rrtb_msphere { /* moving_sphere.h:21-25 */
    float center0[3], center1[3];
    float time0, time1;
    float radius;
    int32_t material;
} rrtb_msphere;

typedef struct rrtb_triangle { /* world-space, already instanced (scene.h:157-170); CCW, triangle.h:5-8 */
    float v0[3], v1[3], v2[3];
    int32_t material;
} rrtb_triangle;

/* SURVEY 8f4 -- "motion blur for object instances" (the reference's README.md:62 to-do; it has no such
 * primitive, the model below follows its moving_sphere.h:27-30): a triangle of an instance whose pose changes
 * between time0 and time1.  Vertices are given at time0; until time1 vertex 0 moves by `delta`, vertex 1 by
 * delta + extra1 and vertex 2 by delta + extra2, each linearly in time -- the keyframe interpolation renderers use
 * for transformation motion blur.  extra1 = extra2 = 0 is a pure translation (scene line `mobj`); an instance that
 * rotates or scales between two poses (scene line `kobj`) has non-zero extras.  The library works on
 *   rate[k]  = delta[k] / (time1 - time0)              base[k]  = fma(-rate[k],  time0, v0[k])            (float)
 *   rate1[k] = extra1[k] / (time1 - time0)             base1[k] = fma(-rate1[k], time0, v1[k] - v0[k])
 *   rate2[k] = extra2[k] / (time1 - time0)             base2[k] = fma(-rate2[k], time0, v2[k] - v0[k])
 *   v0(t) = fma(rate, t, base);  e1(t) = fma(rate1, t, base1);  e2(t) = fma(rate2, t, base2);  v1 = v0 + e1, v2 = v0 + e2
 * (a zero rate keeps its base exactly).  The box spans the camera's shutter interval, as a moving sphere's does
 * (rrt.cu:169): motion is linear, so the two end poses bound every pose in between.  The face normal is that of the
 * pose at the ray's time.  Object ids of moving triangles follow the static triangles'. */
typedef struct rrtb_mtriangle {
    float v0[3], v1[3], v2[3];
    float delta[3];
    float time0, time1;
    int32_t material;
    float extra1[3], extra2[3];
} rrtb_mtriangle;

/* ---- context ------------------------------------------------------------------------------- */

typedef struct rrtb_ctx rrtb_ctx;

int rrtb_abi_version(void);

/* Replaces `-D <n>` + cudaSetDevice (main.cpp:107-110) and the implicit context of Rrt::render. */
int rrtb_create(rrtb_ctx **out, int device);
/* Replaces ~Rrt (rrt.cu:336-342) without the cudaDeviceReset. */
void rrtb_destroy(rrtb_ctx *ctx);
/* Last error text for this context (never NULL). ctx may be NULL: returns the last create error. */
const char *rrtb_last_error(const rrtb_ctx *ctx);
/* Device facts used by `-q` (main.cpp:13-30) and by bench.py. out[0]=SM count, out[1]=max SM clock kHz,
 * out[2]=L2 bytes, out[3]=cc major*10+minor. */
int rrtb_device_info(rrtb_ctx *ctx, int64_t *out4, char *name, int name_len);

/* ---- scene upload + acceleration structure ---------------------------------------------------
 * Replaces the staging copies (rrt.cu:217-247), create_world<<<1,1>>> (rrt.cu:124-174,266) and the
 * single-thread recursive bvh_node build (bvh.h:81-159).  Object ids follow the reference's
 * insertion order: spheres, moving spheres, triangles (rrt.cu:151-164).  With use_bvh != 0 a
 * GPU LBVH (30-bit Morton codes, radix sort, Karras hierarchy, bottom-up refit) is built on the
 * device; with use_bvh == 0 (`-b`) rays scan the flat primitive list (hittable_list.h:95-117).
 * Moving-sphere boxes span [camera.time0, camera.time1] (rrt.cu:169, moving_sphere.h:60-66).
 * One deliberate deviation: sphere boxes use |radius|.  The reference's center -+ radius (sphere.h:60-64) is an
 * inverted box for the negative radii the book uses for hollow glass, and its bvh can then lose the sphere while
 * `-b` renders it; here tree and scan agree.  For radius >= 0 the boxes equal the reference's bit for bit.
 * Every argument is validated before the loaded scene is touched: a rejected call leaves it renderable. */
int rrtb_scene_set(rrtb_ctx *ctx, const rrtb_camera *cam, const rrtb_material *materials, int n_materials,
                   const rrtb_sphere *spheres, int n_spheres, const rrtb_msphere *mspheres, int n_mspheres,
                   const rrtb_triangle *triangles, int n_triangles, int use_bvh);
/* Stage moving triangles (SURVEY 8f4) for the NEXT rrtb_scene_set / rrtb_scene_upload on this context, which
 * consumes them (a later rrtb_scene_set without a new staging call has none).  n == 0 clears the stage. */
int rrtb_scene_stage_moving_triangles(rrtb_ctx *ctx, const rrtb_mtriangle *mtriangles, int n_mtriangles);
/* Stage a constant background for the NEXT rrtb_scene_set / rrtb_scene_upload on this context, with the same staging
 * rule: a segment that leaves the scene adds throughput x rgb3 instead of the reference's sky (rrt.cu:68-75).
 * rgb3 == NULL clears the stage; a rrtb_scene_set without a staged background renders with the sky, bit for bit. */
int rrtb_scene_stage_background(rrtb_ctx *ctx, const float *rgb3);
/* Replace only the camera (animation frames that differ in the camera only; SURVEY f2).  The primitives stay on the
 * device.  If the scene has moving primitives and the shutter interval changed (their boxes span it, rrt.cu:169), or
 * the camera moved farther from the origin than the one the traversal boxes were padded for, the LBVH is rebuilt on
 * the device from the retained scene (stats.seconds_build reports it); otherwise nothing is rebuilt. */
int rrtb_camera_set(rrtb_ctx *ctx, const rrtb_camera *cam);

/* ---- render ------------------------------------------------------------------------------------
 * Replaces render_init + cuda_render (rrt.cu:81-122, launched rrt.cu:289-298) and ray_color
 * (rrt.cu:42-79). */

enum { RRTB_SHARD_TILES = 0, RRTB_SHARD_SAMPLES = 1 };
/* kernel scheduling (same image bit for bit either way; DESIGN.md "scheduling shoot-out"):
 *   RRTB_SCHED_AUTO    the library's default (currently the pool scheduler)
 *   RRTB_SCHED_SIMPLE  persistent threads, one path per lane, the warp syncs at every segment
 *   RRTB_SCHED_POOL    persistent threads, per-warp pool of paths in shared memory: lanes refill as soon as
 *                      their traversal ends, shading runs 32 wide (rrtb_render_pool.cuh) */
enum { RRTB_SCHED_AUTO = 0, RRTB_SCHED_SIMPLE = 1, RRTB_SCHED_POOL = 2 };
/* arithmetic of the integrator = the reference's two builds (rtweekend.h:20-28, Makefile:32-37):
 *   RRTB_PRECISION_F32  `rrt`  (-DUSE_FLOAT): float rays / shading, intersection kernels exact to 2.2e-6 (default)
 *   RRTB_PRECISION_F64  `rrtd` (FP_T = double): rays, hit points, normals, scattering and throughput in double, on
 *                       the same pool scheduler (RRTB_SCHED_SIMPLE and the flat scan: one path per lane).  Same
 *                       Philox streams. */
enum { RRTB_PRECISION_F32 = 0, RRTB_PRECISION_F64 = 1 };

typedef struct rrtb_render_params {
    int32_t width, height;     /* -w -h   (main.cpp:56-57) */
    int32_t spp;               /* -s      (main.cpp:58); 1 <= spp <= 2^23.  Each sample's radiance is clamped to
                                 C = min(2^20, 2^(23 - ceil(log2 spp))) before the 2^40 fixed-point sum, so no pixel
                                 sum passes 2^63 whatever the albedos; C >= 1 never clips radiance <= 1 */
    int32_t max_depth;         /* -d      (main.cpp:66)    */
    uint64_t seed;             /* Philox key; the reference's seed constant is 1984 (rrt.cu:88) */
    int32_t rank, world;       /* this context renders shard `rank` of `world` (1 GPU: 0,1) */
    int32_t shard_mode;        /* RRTB_SHARD_TILES: interleaved 8x4-pixel tiles; RRTB_SHARD_SAMPLES: sample ranges */
    int32_t count_rays;        /* != 0: also count ray segments (stats.rays); same image either way */
    int32_t scheduler;         /* RRTB_SCHED_* */
    int32_t precision;         /* RRTB_PRECISION_* */
} rrtb_render_params;

typedef struct rrtb_stats {
    double seconds_render; /* device time of the render kernel(s), CUDA events */
    double seconds_build;  /* device time of the last rrtb_scene_set (upload + LBVH) */
    double seconds_resolve;/* fixed-point -> float conversion + device->host copy (rrtb_render only) */
    uint64_t rays;         /* ray segments traced (closest-hit queries), if count_rays */
    uint64_t paths;        /* camera paths = pixels_in_shard * spp */
    uint64_t box_tests;    /* counting build only: slab tests, */
    uint64_t sphere_tests; /*   sphere / moving-sphere / triangle tests and */
    uint64_t msphere_tests;
    uint64_t triangle_tests;
    uint64_t hits;         /*   segments that hit something (SURVEY 8d: V_box, V_sph, V_msph, V_tri, h) */
    int32_t kernel_launches;
    int32_t reserved;
} rrtb_stats;

/* Host-buffer entry point (what Rrt::render returns, rrt.h:34): renders this context's shard and
 * writes 3*W*H floats (RGB sums) to the HOST buffer out_rgb. Pixels outside the shard are 0. */
int rrtb_render(rrtb_ctx *ctx, const rrtb_render_params *p, float *out_rgb, rrtb_stats *stats);
/* The same render handed back as DOUBLE sums -- what the reference's `rrtd` build returns (FP_T = double,
 * rtweekend.h:20-28; Makefile:36-37).  A 64-bit fixed-point accumulator converts to double exactly while it is below
 * 2^53 (a pixel sum below 8192 at 2^40 per unit of radiance), and is rounded once above that; this is the framebuffer
 * of the `rrtd` drop-in; rays, RNG and intersection arithmetic are those of rrtb_render. */
int rrtb_render_f64(rrtb_ctx *ctx, const rrtb_render_params *p, double *out_rgb, rrtb_stats *stats);

/* ---- first-hit AOVs (arbitrary output variables: denoiser guides, compositing) ------------------------------------
 * For each pixel and sample s = 0 .. spp-1 the sample's PRIMARY SEGMENT: the camera ray of the beauty render (same
 * Philox streams, lens sample and shutter time) and one closest-hit query with t_min = 0.001.  So the AOVs of samples
 * 0 .. k-1 are those of the first segments of the beauty render's samples 0 .. k-1, whatever spp either uses.
 * Per sample, on a hit / a miss:
 *   albedo    the material's attenuation clamped per channel to [0, 1]: lambertian and metal the albedo, dielectric
 *             (1, 1, 1), RRTB_DIFFUSE_LIGHT its Le                                                  / 0
 *   normal    the hit record's face-forwarded normal (the one shading uses, against the ray)        / 0
 *   depth     Euclidean distance from the ray origin to the hit point, t |d|                        / not counted
 *   coverage  1                                                                                      / 0
 * A miss reports 0, not the sky or the background: coverage tells where the background shows.  Per pixel the outputs
 * are float means: albedo, normal and coverage the sum over the spp samples / spp, depth the sum over the samples that
 * hit / their count (0 if none hit).  Each sum is a double accumulated in sample order 0 .. spp-1 (a miss leaves it as
 * it is), divided once (correctly rounded) and rounded once to float.  The per-sample values are the integrator's:
 * RRTB_PRECISION_F32 float t, normal and distance (sqrt and fma correctly rounded) widened to double when added,
 * RRTB_PRECISION_F64 double throughout.  So the buffers do not depend on the grid, the scheduling, tree or flat scan,
 * or the tile shard. */
/* first-hit AOVs of the shard (p->rank, p->world) of a W x H image: HOST float buffers, bottom-up like rrtb_render;
 * albedo3 / normal3 = 3*W*H, depth / coverage = W*H; pixels outside the shard are 0.  p->precision picks the integrator;
 * p->max_depth and p->scheduler are ignored; p->shard_mode must be RRTB_SHARD_TILES.  stats: seconds_render is the AOV
 * kernel's device time, paths and (count_rays) rays the primary segments, hits those that hit. */
int rrtb_render_aov(rrtb_ctx *ctx, const rrtb_render_params *p, float *albedo3, float *normal3, float *depth,
                    float *coverage, rrtb_stats *stats);

/* Device-resident entry points (used by the multi-GPU host and bench.py):
 *   d_accum : DEVICE pointer (this GPU's memory, or a peer GPU's mapped over NVLink) to 3*W*H
 *             uint64 fixed-point accumulators (value * 2^40), pre-zeroed by the caller.  The kernel
 *             only ever ADDS (64-bit integer atomics), so several GPUs may target one buffer.
 * rrtb_render_device enqueues on the context stream and synchronises before returning. */
int rrtb_render_device(rrtb_ctx *ctx, const rrtb_render_params *p, uint64_t *d_accum, rrtb_stats *stats);
/* d_out_rgb[k] = float(d_accum[k] * 2^-40), k < n   (device pointers) */
int rrtb_resolve_device(rrtb_ctx *ctx, const uint64_t *d_accum, float *d_out_rgb, size_t n);
/* sum 64-bit accumulators: d_dst[k] += d_src[k] (device pointers; d_src may be a peer mapping) */
int rrtb_accumulate_device(rrtb_ctx *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t n);

/* ---- multi-GPU: ONE image over the GPUs of one box (NVLink 5 / NVSwitch) ---------------------------------------
 * The reference renders on one device (`-D n`, main.cpp:107-110); BASELINE north_star asks for tile / sample
 * sharding with the combine over NVLink.  Rank 0 (the OWNER) holds the frame.  Every rank renders its shard into
 * its own accumulator, and its epilogue kernel then writes into the owner's memory directly:
 *   RRTB_SHARD_TILES    the rank's tiles, resolved to 3 floats (or doubles) per pixel, STORED into the owner's frame:
 *                       tiles are disjoint, so there is no reduction and no zero-fill; 12 B/pixel/world cross the link
 *   RRTB_SHARD_SAMPLES  the rank's 64-bit partial sums ADDED into the owner's sum buffer (integer atomics: the image
 *                       does not depend on arrival order); the owner resolves at download time
 * Ranks > 0 reach the owner's memory through a peer mapping: rrtb_frame_attach inside one process (the drop-in's
 * `-G n`), rrtb_frame_export -> (any byte transport, e.g. a torch.distributed broadcast) -> rrtb_frame_import across
 * processes (one process per GPU).  The caller orders the phases: all ranks' rrtb_render_shard have returned (a
 * barrier between processes) before the owner's rrtb_frame_download, and the download has returned before the next
 * frame's shards are rendered. */
#define RRTB_FRAME_HANDLE_BYTES 192
/* owner: allocate (or re-use) the frame for width x height; frame_f64 != 0 = double sums (the `rrtd` framebuffer) */
int rrtb_frame_create(rrtb_ctx *ctx, int width, int height, int frame_f64);
int rrtb_frame_export(rrtb_ctx *ctx, void *handle /* RRTB_FRAME_HANDLE_BYTES */);
int rrtb_frame_import(rrtb_ctx *ctx, const void *handle);
int rrtb_frame_attach(rrtb_ctx *ctx, rrtb_ctx *owner); /* same process; enables peer access ctx -> owner */
int rrtb_frame_detach(rrtb_ctx *ctx);
/* render shard (p->rank, p->world, p->shard_mode) and run the epilogue into the owner's frame; returns when this
 * rank's stores have landed */
int rrtb_render_shard(rrtb_ctx *ctx, const rrtb_render_params *p, rrtb_stats *stats);
/* owner: frame -> host (3*W*H floats, or doubles for an f64 frame).  A destination from rrtb_host_alloc is written
 * by DMA directly; a pageable one goes through pinned staging. */
int rrtb_frame_download(rrtb_ctx *ctx, int shard_mode, void *out_rgb);
/* One process driving n devices (`rrt -G n`): ctxs[0] owns the frame, every context has the scene loaded; all shards
 * are enqueued before any is waited for.  p->rank / p->world are ignored (rank i = ctxs[i], world = n). */
int rrtb_render_group(rrtb_ctx *const *ctxs, int n, const rrtb_render_params *p, int frame_f64, void *out_rgb,
                      rrtb_stats *stats);
/* Pinned (page-locked, portable) host memory for framebuffers and scene arrays: copies to and from it are DMA. */
void *rrtb_host_alloc(size_t bytes);
void rrtb_host_free(void *p);

/* Measurement aid (no reference counterpart; SURVEY 8d): the FP32-issue roofline denominator measured on
 * THIS device -- lane-instructions per second of an FFMA-only loop and of an FFMA+FMNMX (slab-test) mix. */
int rrtb_probe_issue_rate(rrtb_ctx *ctx, double *ffma_lane_instr_per_s, double *mix_lane_instr_per_s);

/* ---- test hooks (parity tests call the same device code the render kernel inlines) ----------- */

/* Closest hit for explicit rays. rays7 = (origin xyz, direction xyz, time) per ray, HOST pointers.
 * mode 0: flat scan (hittable_list.h:95-117 semantics), mode 1: LBVH traversal.
 * id[i] = object id or -1; t[i] = ray parameter; rec7 (optional, may be NULL) = p(3), normal(3), front. */
int rrtb_trace_closest(rrtb_ctx *ctx, const float *rays7, int n, float t_min, int mode, int32_t *id, float *t,
                       float *rec7);
/* The same for the double integrator (RRTB_PRECISION_F64): double rays in, double t / record out. */
int rrtb_trace_closest_f64(rrtb_ctx *ctx, const double *rays7, int n, double t_min, int mode, int32_t *id, double *t,
                           double *rec7);
/* Primary rays exactly as the render kernel generates them (camera.h:31-38, rrt.cu:112-114) for
 * pixel indices pix[k] (= j*W+i) and sample index s. */
int rrtb_camera_rays(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *pix, int n, int sample,
                     float *rays7);
int rrtb_camera_rays_f64(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *pix, int n, int sample,
                         double *rays7);
/* LBVH introspection (all HOST pointers, any may be NULL):
 *   morton[n]            30-bit code of primitive i (object-id order)
 *   perm[n]              sorted position k -> object id
 *   left/right[n-1]      children of internal node i: >=0 internal node, <0 leaf ~k (sorted position)
 *   parent[2n-1]         parent of internal node i (i<n-1) / of leaf k (n-1+k); root's parent = -1
 *   node_box[6*(n-1)]    min xyz, max xyz of internal node i
 *   prim_box[6*n]        min xyz, max xyz of primitive i (object-id order)                       */
int rrtb_bvh_size(rrtb_ctx *ctx, int32_t *n_prims);
int rrtb_bvh_download(rrtb_ctx *ctx, uint32_t *morton, uint32_t *perm, int32_t *left, int32_t *right,
                      int32_t *parent, float *node_box, float *prim_box);
/* The traversal tree the render kernels walk: the 4-wide collapse of the canonical LBVH above (greedy by surface
 * area); *width = 4.  32 floats per node: c.x[4] c.y[4] c.z[4] h.x[4] h.y[4] h.z[4] (padded child boxes as centre /
 * half extent; on the device the half extents are fp16 rounded up and a node is 96 bytes -- this call hands them back
 * widened to float), 4 child refs as int bits, 4 unused.  Child ref >= 0: node index; < 0: ~((sorted position << 2) |
 * primitive type); an unused child slot has h = -inf.  Node 0 is the root; a parent always precedes its children.
 * Test hook: the tree is derived data (closest hit does not depend on it); it is checked for being a partition of
 * the primitives whose boxes enclose them (tests/test_gpu_edge_cases.py) and, raw, word for word against the CPU
 * reference of the build (tests/test_wide_tree.py). */
int rrtb_wide_size(rrtb_ctx *ctx, int32_t *n_nodes, int32_t *width);
int rrtb_wide_download(rrtb_ctx *ctx, float *nodes, int32_t max_nodes);
/* The same nodes as the device holds them, word for word: 24 uint32 per node (rrtb_device.cuh "Traversal node": float
 * centres, fp16 half-extent pairs rounded up, refs, 2 zero words) or, in scenes traversed through motion nodes, 40 per
 * node ("Motion node": centres and half extents at both ends of the shutter).  *words_per_node (may be NULL) gets 24 or
 * 40; `words` holds max_nodes nodes of that size.  Node indices are the build's own (atomic) numbering. */
int rrtb_wide_download_raw(rrtb_ctx *ctx, uint32_t *words, int32_t max_nodes, int32_t *words_per_node);
/* Philox4x32-10 known-answer hook: out[4*i..] = philox(ctr[4*i..], key) computed on the device. */
int rrtb_philox(rrtb_ctx *ctx, const uint32_t *ctr4, int n, uint32_t key0, uint32_t key1, uint32_t *out4);
/* material::scatter (material.h:21-32,50-57,76-96) on the device for explicit inputs.
 * in16 per item : ray o(3) d(3) time, p(3), n(3) (face-forwarded), front, material index, unused
 * rnd4 per item : the Philox block (4 x uint32) the kernel would have drawn for this bounce
 * out8 per item : scattered direction(3), attenuation(3), scattered(0/1), unused                  */
int rrtb_scatter(rrtb_ctx *ctx, const float *in16, const uint32_t *rnd4, int n, float *out8);
int rrtb_scatter_f64(rrtb_ctx *ctx, const double *in16, const uint32_t *rnd4, int n, double *out8);

/* ---- host side of the drop-in (C++ inside the same library; no GPU needed) -------------------
 * Scene-file parser with the reference grammar and quirks (scene.h:212-452, SURVEY Appendix A). */

typedef struct rrtb_scene rrtb_scene;

/* Grammar EXTENSIONS (SURVEY 8f4 and lights; lines the reference ignores silently, like any unknown prefix, or, for
 * an unknown material type, rejects with exit code 3):
 *   mobj <obj index> <material> <dx> <dy> <dz> <time0> <time1> [t x y z | s x y z | r deg x y z]...
 * = `obj` (scene.h:387-427) whose instance, placed by the transforms at time0, translates by (dx, dy, dz) until
 * time1 -- the instance counterpart of `msphere c0 c1 time0 time1 r material`;
 *   kobj <obj index> <material> <time0> <time1> [transforms of the pose at time0]... / [transforms of the pose at time1]...
 * = an instance KEYFRAMED between two poses (any mix of translation, rotation and scale; the word `/` separates the
 * two transform lists): every vertex moves linearly from its place in the first pose to its place in the second;
 *   material <name> diffuse_light <r> <g> <b>
 * = an emitter (RRTB_DIFFUSE_LIGHT) of radiance (r, g, b);
 *   background <r> <g> <b>
 * = the constant background of rrtb_scene_stage_background; the LAST background line wins, as for `camera`.
 * On failure *out = NULL and *ref_exit_code (optional) receives the exit code the reference would
 * have used (1, 2, 3 or 4); err/err_len (optional) receive the reference's message. */
int rrtb_scene_parse_file(const char *path, int image_width, int image_height, rrtb_scene **out,
                          int *ref_exit_code, char *err, int err_len);
void rrtb_scene_free(rrtb_scene *s);
/* counts[6] = materials, spheres, moving spheres, triangles (flattened), objs, obj instances */
int rrtb_scene_counts(const rrtb_scene *s, int32_t *counts6);
const rrtb_camera *rrtb_scene_camera(const rrtb_scene *s);
const rrtb_material *rrtb_scene_materials(const rrtb_scene *s);
const rrtb_sphere *rrtb_scene_spheres(const rrtb_scene *s);
const rrtb_msphere *rrtb_scene_mspheres(const rrtb_scene *s);
const rrtb_triangle *rrtb_scene_triangles(const rrtb_scene *s);
/* moving triangles of `mobj` instances (grammar extension, see rrtb_scene_parse_file) */
int rrtb_scene_mtriangle_count(const rrtb_scene *s);
const rrtb_mtriangle *rrtb_scene_mtriangles(const rrtb_scene *s);
/* 1 and rgb3 = the file's `background` (grammar extension), or 0 (rgb3 untouched) if it has none: the sky */
int rrtb_scene_background(const rrtb_scene *s, float *rgb3);
/* rrtb_scene_set with a parsed scene (its moving triangles and background staged first). */
int rrtb_scene_upload(rrtb_ctx *ctx, const rrtb_scene *s, int use_bvh);
/* camera.h:8-29 in the reference's float arithmetic. */
int rrtb_camera_derive(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov,
                       float aspect_ratio, float aperture, float focus_dist, float time0, float time1,
                       rrtb_camera *out);
/* color.h:8-23 + the vertical flip of main.cpp:150-163: rgb_sum (bottom-up sums) -> rgb8 (top-down). */
int rrtb_tonemap_rgb8(const float *rgb_sum, int width, int height, int spp, uint8_t *rgb8);
/* the same in the double build's arithmetic (FP_T = double in color.h:8-23) */
int rrtb_tonemap_rgb8_f64(const double *rgb_sum, int width, int height, int spp, uint8_t *rgb8);
/* PNG writer used where the reference calls stbi_write_png (main.cpp:164). */
int rrtb_write_png(const char *path, int width, int height, const uint8_t *rgb8);
/* PFM (Portable Float Map): channels 3 ("PF") or 1 ("Pf"), little endian (scale -1.0); PFM rows run bottom to top,
 * which is this library's framebuffer order, so no flip */
int rrtb_write_pfm(const char *path, int width, int height, int channels, const float *data);

#ifdef __cplusplus
}
#endif
#endif /* RRTB_H */
