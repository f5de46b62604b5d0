// rrtb_api.cu -- the C ABI of librrtb200.so (include/rrtb.h): context, scene upload, render, test hooks.
// The reference interfaces each entry point replaces are cited in include/rrtb.h.
#include "rrtb_internal.h"

#include <math.h>
#include <stdio.h>
#include <string.h>

#include <mutex>

namespace rrtb {

static std::string g_create_error;
static std::mutex g_mutex;

int cuda_fail(rrtb_ctx *ctx, cudaError_t e, const char *expr, const char *file, int line)
{
    // same wording as the reference's check_cuda (rrt.cu:31-40), plus the CUDA error string
    char buf[512];
    snprintf(buf, sizeof(buf), "CUDA error = %u at %s:%d '%s' (%s)", (unsigned)e, file, line, expr,
             cudaGetErrorString(e));
    if (ctx) ctx->err = buf;
    else {
        std::lock_guard<std::mutex> lk(g_mutex);
        g_create_error = buf;
    }
    cudaGetLastError(); // clear the sticky-less error state
    return RRTB_ERR_CUDA;
}

int read_back(rrtb_ctx *ctx, void *dst, const void *d_src, size_t bytes)
{
    RRTB_CUDA(ctx, cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

static int invalid(rrtb_ctx *ctx, const char *msg)
{
    if (ctx) ctx->err = msg;
    return RRTB_ERR_INVALID;
}

static int require_scene(rrtb_ctx *ctx, const char *msg)
{
    if (ctx->has_scene) return RRTB_OK;
    ctx->err = msg;
    return RRTB_ERR_NO_SCENE;
}

static void frame_drop_mapping(rrtb_ctx *ctx)
{
    if (ctx->peer_is_ipc) {
        if (ctx->peer_frame) cudaIpcCloseMemHandle(ctx->peer_frame);
        if (ctx->peer_sum) cudaIpcCloseMemHandle(ctx->peer_sum);
    }
    ctx->peer_frame = nullptr;
    ctx->peer_sum = nullptr;
    ctx->peer_is_ipc = false;
}

// Builds the acceleration structure from the raw scene in d_stage and marks the scene renderable.  `upload()` enqueues
// what the build reads that is not on the device yet; stats.seconds_build times it together with the build.
template <typename Upload>
static int build_scene(rrtb_ctx *ctx, Upload &&upload)
{
    cudaStream_t st = ctx->stream;
    ctx->has_scene = false; // until the build below has succeeded
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
    int rc = upload();
    if (rc || (rc = prepare_and_build(ctx))) return rc;
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
    // did the collapse kernel's work list drain (CollapseState::stuck == 0)?  Read back behind the build into pinned
    // memory: it costs no synchronisation of its own
    if ((rc = ctx->h_state.reserve(ctx, 4))) return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(ctx->h_state, ctx->d_collapse, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
    RRTB_CUDA(ctx, cudaStreamSynchronize(st)); // the caller's host arrays may go away after this
    float ms = 0.f;
    RRTB_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->seconds_build = ms * 1e-3;
    if (ctx->h_state[3]) {
        ctx->err = "internal error: the 4-wide collapse did not terminate (inconsistent tree)";
        return RRTB_ERR_CUDA;
    }
    ctx->has_scene = true;
    return RRTB_OK;
}

} // namespace rrtb

rrtb_ctx::~rrtb_ctx()
{
    rrtb::frame_drop_mapping(this);
    for (cudaEvent_t e : {ev0, ev1, ev2, ev3, ev_copy[0], ev_copy[1]})
        if (e) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
}

using namespace rrtb;

extern "C" {

int rrtb_abi_version(void) { return RRTB_ABI_VERSION; }

int rrtb_create(rrtb_ctx **out, int device)
{
    if (!out) return RRTB_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        std::lock_guard<std::mutex> lk(g_mutex);
        g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) +
                         "); librrtb200 has no CPU fallback";
        cudaGetLastError();
        return RRTB_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) {
        std::lock_guard<std::mutex> lk(g_mutex);
        g_create_error = "device index out of range";
        return RRTB_ERR_NO_DEVICE;
    }
    rrtb_ctx *ctx = new rrtb_ctx();
    ctx->device = device;
    auto fail = [&](int rc) { // the destructor releases what was created so far
        {
            std::lock_guard<std::mutex> lk(g_mutex);
            g_create_error = ctx->err;
        }
        delete ctx;
        return rc;
    };
#define CREATE_CUDA(expr)                                                            \
    do {                                                                             \
        cudaError_t _e = (expr);                                                     \
        if (_e != cudaSuccess) return fail(cuda_fail(ctx, _e, #expr, __FILE__, __LINE__)); \
    } while (0)
    CREATE_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CREATE_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CREATE_CUDA(cudaEventCreate(&ctx->ev0));
    CREATE_CUDA(cudaEventCreate(&ctx->ev1));
    CREATE_CUDA(cudaEventCreate(&ctx->ev2));
    CREATE_CUDA(cudaEventCreate(&ctx->ev3));
#undef CREATE_CUDA
    if (int rc = ctx->d_counters.reserve(ctx, 8)) return fail(rc);
    *out = ctx;
    return RRTB_OK;
}

void rrtb_destroy(rrtb_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    delete ctx;
}

const char *rrtb_last_error(const rrtb_ctx *ctx)
{
    if (ctx) return ctx->err.c_str();
    static thread_local std::string copy;
    std::lock_guard<std::mutex> lk(g_mutex);
    copy = g_create_error;
    return copy.c_str();
}

int rrtb_device_info(rrtb_ctx *ctx, int64_t *out4, char *name, int name_len)
{
    if (!ctx) return RRTB_ERR_INVALID;
    cudaDeviceProp prop;
    RRTB_CUDA(ctx, cudaGetDeviceProperties(&prop, ctx->device));
    if (out4) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
        out4[0] = prop.multiProcessorCount;
        out4[1] = khz;
        out4[2] = prop.l2CacheSize;
        out4[3] = prop.major * 10 + prop.minor;
    }
    if (name && name_len > 0) {
        strncpy(name, prop.name, (size_t)name_len - 1);
        name[name_len - 1] = 0;
    }
    return RRTB_OK;
}

// Motion nodes (rrtb_device.cuh) interpolate the child boxes at the ray's time: tighter boxes, but 160-byte nodes and a
// third more arithmetic per visit.  A handful of moving primitives does not pay for that (scenes/test3.txt, 3 moving
// spheres: 26.1 Grays/s with motion nodes, 28.5 with shutter-spanning boxes), many do (64 fast spheres: less than half the
// exact tests per ray), so they are used from 8 moving primitives on, under an open shutter.
static bool use_motion_nodes(int n_moving, const rrtb_camera *cam) { return n_moving >= 8 && cam->time0 != cam->time1; }

int rrtb_scene_stage_moving_triangles(rrtb_ctx *ctx, const rrtb_mtriangle *mtriangles, int n_mtriangles)
{
    if (!ctx || n_mtriangles < 0 || (n_mtriangles > 0 && !mtriangles)) return RRTB_ERR_INVALID;
    for (int i = 0; i < n_mtriangles; ++i)
        if (!(mtriangles[i].time1 != mtriangles[i].time0)) return invalid(ctx, "moving triangle needs time0 != time1");
    ctx->staged_mtriangles.assign(mtriangles, mtriangles + n_mtriangles);
    return RRTB_OK;
}

int rrtb_scene_stage_background(rrtb_ctx *ctx, const float *rgb3)
{
    if (!ctx) return RRTB_ERR_INVALID;
    ctx->staged_background = rgb3 != nullptr;
    for (int k = 0; k < 3; ++k) ctx->staged_bg[k] = rgb3 ? rgb3[k] : 0.f;
    return RRTB_OK;
}

int rrtb_scene_set(rrtb_ctx *ctx, const rrtb_camera *cam, const rrtb_material *materials, int n_materials,
                   const rrtb_sphere *spheres, int n_spheres, const rrtb_msphere *mspheres, int n_mspheres,
                   const rrtb_triangle *triangles, int n_triangles, int use_bvh)
{
    if (!ctx) return RRTB_ERR_INVALID;
    // staged moving triangles (SURVEY 8f4) and background belong to this call whether it succeeds or not
    std::vector<rrtb_mtriangle> mtri;
    mtri.swap(ctx->staged_mtriangles);
    const bool background = ctx->staged_background;
    const float bg[3] = {ctx->staged_bg[0], ctx->staged_bg[1], ctx->staged_bg[2]};
    ctx->staged_background = false;
    const int n_mtriangles = (int)mtri.size();
    if (!cam || !materials || n_materials <= 0) return invalid(ctx, "scene needs a camera and at least one material");
    if (n_spheres < 0 || n_mspheres < 0 || n_triangles < 0) return invalid(ctx, "negative primitive count");
    const long long n_ll = (long long)n_spheres + n_mspheres + n_triangles + n_mtriangles;
    if (n_ll <= 0) return invalid(ctx, "scene has no objects");
    if (n_ll >= (1ll << 28)) return invalid(ctx, "too many primitives (limit 2^28: 32-bit element offsets such as 6 * id)");
    if ((n_spheres && !spheres) || (n_mspheres && !mspheres) || (n_triangles && !triangles))
        return invalid(ctx, "null primitive array");
    const int n = (int)n_ll;
    // everything is validated BEFORE the loaded scene is touched: a rejected call leaves it renderable
    bool emitters = false;
    for (int i = 0; i < n_materials; ++i) {
        if (materials[i].type < RRTB_LAMBERTIAN || materials[i].type > RRTB_DIFFUSE_LIGHT) return invalid(ctx, "unknown material type");
        emitters |= materials[i].type == RRTB_DIFFUSE_LIGHT;
    }
    for (int i = 0; i < n_spheres; ++i)
        if (spheres[i].material < 0 || spheres[i].material >= n_materials) return invalid(ctx, "sphere material index out of range");
    for (int i = 0; i < n_mspheres; ++i) {
        if (mspheres[i].material < 0 || mspheres[i].material >= n_materials) return invalid(ctx, "msphere material index out of range");
        // moving_sphere.h:27-30 divides by (time1 - time0)
        if (!(mspheres[i].time1 != mspheres[i].time0)) return invalid(ctx, "moving sphere needs time0 != time1");
    }
    for (int i = 0; i < n_triangles; ++i)
        if (triangles[i].material < 0 || triangles[i].material >= n_materials) return invalid(ctx, "triangle material index out of range");
    for (int i = 0; i < n_mtriangles; ++i)
        if (mtri[i].material < 0 || mtri[i].material >= n_materials) return invalid(ctx, "moving triangle material index out of range");

    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    ctx->has_scene = false; // until the build below has succeeded
    ctx->cam = *cam;
    ctx->n_materials = n_materials;
    ctx->n_spheres = n_spheres;
    ctx->n_mspheres = n_mspheres;
    ctx->n_triangles = n_triangles;
    ctx->n_mtriangles = n_mtriangles;
    ctx->n_prims = n;
    ctx->use_bvh = use_bvh ? 1 : 0;
    ctx->motion = use_motion_nodes(n_mspheres + n_mtriangles, cam);
    ctx->background = background;
    for (int k = 0; k < 3; ++k) ctx->bg[k] = bg[k];
    ctx->lights = emitters || background;

    int rc;
    const int nb = (n + 255) / 256;
    const int n_seg = (n + 1023) / 1024;
    const size_t b_sph = (sizeof(rrtb_sphere) * (size_t)n_spheres + 15) & ~(size_t)15;
    const size_t b_msph = (sizeof(rrtb_msphere) * (size_t)n_mspheres + 15) & ~(size_t)15;
    const size_t b_tri = (sizeof(rrtb_triangle) * (size_t)n_triangles + 15) & ~(size_t)15;
    const size_t b_mtri = (sizeof(rrtb_mtriangle) * (size_t)n_mtriangles + 15) & ~(size_t)15;
    if ((rc = ctx->d_prim.reserve(ctx, (size_t)3 * n))) return rc;
    if ((rc = ctx->d_prim_info.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_materials.reserve(ctx, (size_t)n_materials))) return rc;
    if ((rc = ctx->d_material_type.reserve(ctx, (size_t)n_materials))) return rc;
    if ((rc = ctx->d_prim_box.reserve(ctx, (size_t)6 * n))) return rc;
    if ((rc = ctx->d_morton.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_keys.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_keys_tmp.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_left.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_right.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_parent.reserve(ctx, (size_t)2 * n))) return rc;
    if ((rc = ctx->d_node_box.reserve(ctx, (size_t)6 * n))) return rc;
    if ((rc = ctx->d_visit.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_range.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_left2.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_right2.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_parent2.reserve(ctx, (size_t)2 * n))) return rc;
    if ((rc = ctx->d_node_box2.reserve(ctx, (size_t)6 * n))) return rc;
    if ((rc = ctx->d_sah_roots.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_wnodes.reserve(ctx, (size_t)(n_mspheres + n_mtriangles > 0 ? RRTB_MOTION_NODE_F4 : RRTB_NODE_F4) * n))) return rc;
    if (n_mspheres + n_mtriangles > 0) { // room for the end-of-shutter boxes whatever this camera's shutter is (rrtb_camera_set may open it)
        if ((rc = ctx->d_prim_box01.reserve(ctx, (size_t)12 * n))) return rc;
        if ((rc = ctx->d_node_box01.reserve(ctx, (size_t)12 * n))) return rc;
    }
    if ((rc = ctx->d_wq.reserve(ctx, (size_t)n))) return rc;
    if ((rc = ctx->d_collapse.reserve(ctx, (size_t)16))) return rc; // CollapseState, SahState
    if ((rc = ctx->d_leaves.reserve(ctx, (size_t)3 * n))) return rc;
    if ((rc = ctx->d_leaf_info.reserve(ctx, (size_t)n))) return rc;
    if (n_mtriangles > 0) { // edge rates of moving triangles (SURVEY 8f4): two float4 per slot, only for scenes that have them
        if ((rc = ctx->d_prim_ext.reserve(ctx, (size_t)2 * n))) return rc;
        if ((rc = ctx->d_leaf_ext.reserve(ctx, (size_t)2 * n))) return rc;
    }
    if ((rc = ctx->d_reduce.reserve(ctx, (size_t)nb * 7 + 16))) return rc;
    if ((rc = ctx->d_hist.reserve(ctx, (size_t)256 * n_seg + (size_t)(256 * n_seg + 4095) / 4096 + 1))) return rc; // + chunk sums
    if ((rc = ctx->d_stage.reserve(ctx, b_sph + b_msph + b_tri + b_mtri))) return rc;

    // materials -> (albedo.xyz, param) + type
    std::vector<float4> mats((size_t)n_materials);
    std::vector<int> mtypes((size_t)n_materials);
    for (int i = 0; i < n_materials; ++i) {
        const rrtb_material &m = materials[i];
        mats[i] = make_float4(m.albedo[0], m.albedo[1], m.albedo[2], m.param);
        mtypes[i] = m.type;
    }

    // raw structs, staged in one device buffer for k_prepare
    ctx->stage_off[0] = 0;
    ctx->stage_off[1] = b_sph;
    ctx->stage_off[2] = b_sph + b_msph;
    ctx->stage_off[3] = b_sph + b_msph + b_tri;
    return build_scene(ctx, [&]() -> int {
        cudaStream_t st = ctx->stream;
        unsigned char *stage = ctx->d_stage;
        if (n_mtriangles > 0) RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_prim_ext, 0, sizeof(float4) * 2 * (size_t)n, st)); // static primitives: no rates
        RRTB_CUDA(ctx, cudaMemcpyAsync(ctx->d_materials, mats.data(), sizeof(float4) * n_materials, cudaMemcpyHostToDevice, st));
        RRTB_CUDA(ctx, cudaMemcpyAsync(ctx->d_material_type, mtypes.data(), sizeof(int) * n_materials, cudaMemcpyHostToDevice, st));
        if (n_spheres)
            RRTB_CUDA(ctx, cudaMemcpyAsync(stage, spheres, sizeof(rrtb_sphere) * (size_t)n_spheres, cudaMemcpyHostToDevice, st));
        if (n_mspheres)
            RRTB_CUDA(ctx, cudaMemcpyAsync(stage + b_sph, mspheres, sizeof(rrtb_msphere) * (size_t)n_mspheres, cudaMemcpyHostToDevice, st));
        if (n_triangles)
            RRTB_CUDA(ctx, cudaMemcpyAsync(stage + b_sph + b_msph, triangles, sizeof(rrtb_triangle) * (size_t)n_triangles,
                                           cudaMemcpyHostToDevice, st));
        if (n_mtriangles)
            RRTB_CUDA(ctx, cudaMemcpyAsync(stage + b_sph + b_msph + b_tri, mtri.data(), sizeof(rrtb_mtriangle) * (size_t)n_mtriangles,
                                           cudaMemcpyHostToDevice, st));
        return RRTB_OK;
    });
}

int rrtb_camera_set(rrtb_ctx *ctx, const rrtb_camera *cam)
{
    if (!ctx || !cam) return RRTB_ERR_INVALID;
    if (int rc = require_scene(ctx, "no scene")) return rc;
    // Two things of the acceleration structure depend on the camera: the boxes of moving primitives span its shutter
    // interval (rrt.cu:169), and the padding of the traversal boxes scales with the largest coordinate a ray can
    // start from.  When either changes, the LBVH is rebuilt from the raw scene kept on the device (no upload).
    float mag = 0.f;
    for (int k = 0; k < 3; ++k) mag = fmaxf(mag, fabsf(cam->origin[k]) + cam->lens_radius);
    const bool shutter = ctx->n_mspheres + ctx->n_mtriangles > 0 && (cam->time0 != ctx->cam.time0 || cam->time1 != ctx->cam.time1);
    const bool farther = mag > ctx->build_cam_mag;
    ctx->cam = *cam;
    ctx->motion = use_motion_nodes(ctx->n_mspheres + ctx->n_mtriangles, cam);
    if (!(shutter || farther)) return RRTB_OK;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    return build_scene(ctx, [] { return RRTB_OK; }); // the raw scene is on the device already
}

// Device -> host copy of a result.  A pinned destination (rrtb_host_alloc, cudaHostRegister) is written by DMA
// directly; a pageable one is fed through two pinned 4 MB halves so that the copy engine and the host memcpy overlap
// (a plain cudaMemcpy into pageable memory serialises the two).
static int copy_to_host(rrtb_ctx *ctx, void *dst, const void *d_src, size_t bytes)
{
    cudaPointerAttributes at;
    const bool pinned = cudaPointerGetAttributes(&at, dst) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (pinned) {
        RRTB_CUDA(ctx, cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return RRTB_OK;
    }
    const size_t CH = (size_t)4 << 20;
    if (int rc = ctx->h_pinned.reserve(ctx, 2 * CH)) return rc;
    if (!ctx->ev_copy[0]) {
        RRTB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_copy[0], cudaEventDisableTiming));
        RRTB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_copy[1], cudaEventDisableTiming));
    }
    const size_t n_chunks = (bytes + CH - 1) / CH;
    for (size_t k = 0; k <= n_chunks; ++k) {
        if (k < n_chunks) {
            if (k >= 2) RRTB_CUDA(ctx, cudaEventSynchronize(ctx->ev_copy[k & 1])); // (its memcpy below is done too: same thread)
            const size_t len = (k + 1 == n_chunks) ? bytes - k * CH : CH;
            RRTB_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + (k & 1) * CH, (const char *)d_src + k * CH, len,
                                           cudaMemcpyDeviceToHost, ctx->stream));
            RRTB_CUDA(ctx, cudaEventRecord(ctx->ev_copy[k & 1], ctx->stream));
        }
        if (k >= 1) {
            const size_t j = k - 1, len = (j + 1 == n_chunks) ? bytes - j * CH : CH;
            RRTB_CUDA(ctx, cudaEventSynchronize(ctx->ev_copy[j & 1]));
            memcpy((char *)dst + j * CH, ctx->h_pinned + (j & 1) * CH, len);
        }
    }
    return RRTB_OK;
}

static int check_render(rrtb_ctx *ctx, const rrtb_render_params *p)
{
    if (!ctx || !p) return RRTB_ERR_INVALID;
    if (int rc = require_scene(ctx, "render before rrtb_scene_set")) return rc;
    if (p->width < 2 || p->height < 2) return invalid(ctx, "image must be at least 2x2 (u = (i+xi)/(W-1), rrt.cu:112)");
    if (p->spp < 1 || p->max_depth < 0) return invalid(ctx, "spp must be >= 1 and max_depth >= 0");
    if (p->spp > rrtb::MAX_SPP) return invalid(ctx, "spp must be <= 2^23 (64-bit fixed-point pixel sums, rrtb_device.cuh fixed_clamp)");
    if ((long long)p->width * p->height >= (1ll << 28)) return invalid(ctx, "image too large (limit 2^28 pixels)");
    if (p->rank < 0 || p->rank >= (p->world > 1 ? p->world : 1)) return invalid(ctx, "rank out of range (0 <= rank < max(world, 1))");
    if (p->shard_mode != RRTB_SHARD_TILES && p->shard_mode != RRTB_SHARD_SAMPLES) return invalid(ctx, "bad shard_mode");
    if (p->precision != RRTB_PRECISION_F32 && p->precision != RRTB_PRECISION_F64) return invalid(ctx, "bad precision");
    return RRTB_OK;
}

int rrtb_render_device(rrtb_ctx *ctx, const rrtb_render_params *p, uint64_t *d_accum, rrtb_stats *stats)
{
    int rc = check_render(ctx, p);
    if (rc) return rc;
    if (!d_accum) return invalid(ctx, "null accumulator");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    return launch_render(ctx, p, d_accum, stats);
}

int rrtb_resolve_device(rrtb_ctx *ctx, const uint64_t *d_accum, float *d_out_rgb, size_t n)
{
    if (!ctx || !d_accum || !d_out_rgb) return RRTB_ERR_INVALID;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = launch_resolve(ctx, d_accum, d_out_rgb, n);
    if (rc) return rc;
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

int rrtb_accumulate_device(rrtb_ctx *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t n)
{
    if (!ctx || !d_dst || !d_src) return RRTB_ERR_INVALID;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = launch_accumulate(ctx, d_dst, d_src, n);
    if (rc) return rc;
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

static int render_host(rrtb_ctx *ctx, const rrtb_render_params *p, void *out_rgb, rrtb_stats *stats, bool f64)
{
    int rc = check_render(ctx, p);
    if (rc) return rc;
    if (!out_rgb) return invalid(ctx, "null output buffer");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)3 * p->width * p->height;
    if ((rc = ctx->d_accum.reserve(ctx, n)) || (rc = ctx->d_rgb.reserve(ctx, n))) return rc;
    RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_accum, 0, n * sizeof(unsigned long long), ctx->stream));
    rrtb_stats local;
    memset(&local, 0, sizeof(local));
    rc = launch_render(ctx, p, ctx->d_accum, &local);
    if (rc) return rc;
    cudaEvent_t e0 = ctx->ev0, e1 = ctx->ev1;
    RRTB_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    rc = f64 ? launch_resolve(ctx, ctx->d_accum, ctx->d_rgb.get(), n) : launch_resolve(ctx, ctx->d_accum, (float *)ctx->d_rgb.get(), n);
    if (rc) return rc;
    if ((rc = copy_to_host(ctx, out_rgb, ctx->d_rgb, n * (f64 ? sizeof(double) : sizeof(float))))) return rc;
    RRTB_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    RRTB_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
    local.seconds_resolve = ms * 1e-3;
    local.kernel_launches += 1;
    if (stats) *stats = local;
    return RRTB_OK;
}

int rrtb_render(rrtb_ctx *ctx, const rrtb_render_params *p, float *out_rgb, rrtb_stats *stats)
{
    return render_host(ctx, p, out_rgb, stats, false);
}

int rrtb_render_f64(rrtb_ctx *ctx, const rrtb_render_params *p, double *out_rgb, rrtb_stats *stats)
{
    return render_host(ctx, p, out_rgb, stats, true);
}

int rrtb_render_aov(rrtb_ctx *ctx, const rrtb_render_params *p, float *albedo3, float *normal3, float *depth, float *coverage,
                    rrtb_stats *stats)
{
    int rc = check_render(ctx, p);
    if (rc) return rc;
    // a pixel's double sums split over sample shards would not add up to one GPU's bits
    if (p->shard_mode != RRTB_SHARD_TILES) return invalid(ctx, "rrtb_render_aov shards by tiles only (RRTB_SHARD_TILES)");
    if (!albedo3 || !normal3 || !depth || !coverage) return invalid(ctx, "null output buffer");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)p->width * p->height;
    if ((rc = ctx->d_aov.reserve(ctx, 8 * n))) return rc;
    rrtb_stats local;
    memset(&local, 0, sizeof(local));
    if ((rc = launch_aov(ctx, p, ctx->d_aov, &local))) return rc;
    if ((rc = copy_to_host(ctx, albedo3, ctx->d_aov, 3 * n * sizeof(float)))) return rc;
    if ((rc = copy_to_host(ctx, normal3, ctx->d_aov + 3 * n, 3 * n * sizeof(float)))) return rc;
    if ((rc = copy_to_host(ctx, depth, ctx->d_aov + 6 * n, n * sizeof(float)))) return rc;
    if ((rc = copy_to_host(ctx, coverage, ctx->d_aov + 7 * n, n * sizeof(float)))) return rc;
    if (stats) *stats = local;
    return RRTB_OK;
}

// ---- multi-GPU frame (SURVEY 8e) ---------------------------------------------------------------------------------
namespace {
struct FrameHandle { // what crosses the process boundary (RRTB_FRAME_HANDLE_BYTES)
    cudaIpcMemHandle_t frame, sum;
    int32_t width, height, f64, device;
};
static_assert(sizeof(FrameHandle) <= RRTB_FRAME_HANDLE_BYTES, "handle blob too small");
} // namespace

int rrtb_frame_create(rrtb_ctx *ctx, int width, int height, int frame_f64)
{
    if (!ctx) return RRTB_ERR_INVALID;
    if (width < 2 || height < 2 || (long long)width * height >= (1ll << 28)) return invalid(ctx, "bad frame size");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    frame_drop_mapping(ctx);
    const size_t n = (size_t)3 * width * height;
    int rc;
    if ((rc = ctx->d_frame.reserve(ctx, n)) || (rc = ctx->d_sum.reserve(ctx, n))) return rc;
    ctx->frame_w = width;
    ctx->frame_h = height;
    ctx->frame_f64 = frame_f64 ? 1 : 0;
    RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_sum, 0, n * sizeof(unsigned long long), ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

int rrtb_frame_export(rrtb_ctx *ctx, void *handle)
{
    if (!ctx || !handle) return RRTB_ERR_INVALID;
    if (!ctx->d_frame) return invalid(ctx, "rrtb_frame_export before rrtb_frame_create");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    FrameHandle h;
    memset(&h, 0, sizeof(h));
    RRTB_CUDA(ctx, cudaIpcGetMemHandle(&h.frame, ctx->d_frame));
    RRTB_CUDA(ctx, cudaIpcGetMemHandle(&h.sum, ctx->d_sum));
    h.width = ctx->frame_w;
    h.height = ctx->frame_h;
    h.f64 = ctx->frame_f64;
    h.device = ctx->device;
    memset(handle, 0, RRTB_FRAME_HANDLE_BYTES);
    memcpy(handle, &h, sizeof(h));
    return RRTB_OK;
}

int rrtb_frame_import(rrtb_ctx *ctx, const void *handle)
{
    if (!ctx || !handle) return RRTB_ERR_INVALID;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    frame_drop_mapping(ctx);
    FrameHandle h;
    memcpy(&h, handle, sizeof(h));
    if (h.width < 2 || h.height < 2) return invalid(ctx, "bad frame handle");
    // peer mapping of the owner's allocations: loads and stores of this context's kernels go over NVLink
    RRTB_CUDA(ctx, cudaIpcOpenMemHandle(&ctx->peer_frame, h.frame, cudaIpcMemLazyEnablePeerAccess));
    void *sum = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&sum, h.sum, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        cudaIpcCloseMemHandle(ctx->peer_frame);
        ctx->peer_frame = nullptr;
        return cuda_fail(ctx, e, "cudaIpcOpenMemHandle(sum)", __FILE__, __LINE__);
    }
    ctx->peer_sum = (uint64_t *)sum;
    ctx->peer_is_ipc = true;
    ctx->frame_w = h.width;
    ctx->frame_h = h.height;
    ctx->frame_f64 = h.f64;
    return RRTB_OK;
}

int rrtb_frame_attach(rrtb_ctx *ctx, rrtb_ctx *owner)
{
    if (!ctx || !owner || ctx == owner) return RRTB_ERR_INVALID;
    if (!owner->d_frame) return invalid(ctx, "rrtb_frame_attach before the owner's rrtb_frame_create");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    frame_drop_mapping(ctx);
    if (ctx->device != owner->device) {
        int can = 0;
        RRTB_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, owner->device));
        if (!can) return invalid(ctx, "no peer access between the two devices");
        cudaError_t e = cudaDeviceEnablePeerAccess(owner->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(ctx, e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
        cudaGetLastError();
    }
    ctx->peer_frame = owner->d_frame; // unified addressing: the owner's pointers are valid on this device
    ctx->peer_sum = owner->d_sum;
    ctx->peer_is_ipc = false;
    ctx->frame_w = owner->frame_w;
    ctx->frame_h = owner->frame_h;
    ctx->frame_f64 = owner->frame_f64;
    return RRTB_OK;
}

int rrtb_frame_detach(rrtb_ctx *ctx)
{
    if (!ctx) return RRTB_ERR_INVALID;
    cudaSetDevice(ctx->device);
    frame_drop_mapping(ctx);
    return RRTB_OK;
}

// enqueue: zero the own accumulator, render the shard, epilogue into the owner's frame / sum buffer
static int enqueue_shard(rrtb_ctx *ctx, const rrtb_render_params *p)
{
    int rc = check_render(ctx, p);
    if (rc) return rc;
    void *frame = ctx->peer_frame ? ctx->peer_frame : ctx->d_frame;
    uint64_t *sum = ctx->peer_frame ? ctx->peer_sum : ctx->d_sum;
    if (!frame) return invalid(ctx, "no frame: call rrtb_frame_create (owner) or rrtb_frame_import / rrtb_frame_attach first");
    if (p->width != ctx->frame_w || p->height != ctx->frame_h) return invalid(ctx, "render size differs from the frame's");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)3 * p->width * p->height;
    if ((rc = ctx->d_accum.reserve(ctx, n))) return rc;
    RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_accum, 0, n * sizeof(unsigned long long), ctx->stream));
    if ((rc = launch_render(ctx, p, ctx->d_accum, nullptr, true))) return rc;
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
    if (p->shard_mode == RRTB_SHARD_TILES) rc = launch_resolve_tiles(ctx, ctx->d_accum, frame, p, ctx->frame_f64 != 0);
    else rc = launch_accumulate_atomic(ctx, sum, ctx->d_accum, n);
    if (rc) return rc;
    RRTB_CUDA(ctx, cudaEventRecord(ctx->ev3, ctx->stream));
    return RRTB_OK;
}

static int finish_shard(rrtb_ctx *ctx, rrtb_stats *stats)
{
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    rrtb_stats local;
    memset(&local, 0, sizeof(local));
    int rc = finish_render(ctx, &local); // synchronises the stream: the peer stores of the epilogue have landed
    if (rc) return rc;
    float ms = 0.f;
    RRTB_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev2, ctx->ev3));
    local.seconds_resolve = ms * 1e-3;
    local.kernel_launches += 1;
    if (stats) *stats = local;
    return RRTB_OK;
}

int rrtb_render_shard(rrtb_ctx *ctx, const rrtb_render_params *p, rrtb_stats *stats)
{
    if (!ctx || !p) return RRTB_ERR_INVALID;
    int rc = enqueue_shard(ctx, p);
    if (rc) return rc;
    return finish_shard(ctx, stats);
}

int rrtb_frame_download(rrtb_ctx *ctx, int shard_mode, void *out_rgb)
{
    if (!ctx || !out_rgb) return RRTB_ERR_INVALID;
    if (!ctx->d_frame || ctx->peer_frame) return invalid(ctx, "rrtb_frame_download is the owner's call (after rrtb_frame_create)");
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)3 * ctx->frame_w * ctx->frame_h;
    if (shard_mode == RRTB_SHARD_SAMPLES) { // the ranks added their partial sums: resolve them, then clear for the next frame
        int rc = ctx->frame_f64 ? launch_resolve(ctx, ctx->d_sum, ctx->d_frame.get(), n)
                                : launch_resolve(ctx, ctx->d_sum, (float *)ctx->d_frame.get(), n);
        if (rc) return rc;
        RRTB_CUDA(ctx, cudaMemsetAsync(ctx->d_sum, 0, n * sizeof(unsigned long long), ctx->stream));
    }
    else if (shard_mode != RRTB_SHARD_TILES) return invalid(ctx, "bad shard_mode");
    return copy_to_host(ctx, out_rgb, ctx->d_frame, n * (ctx->frame_f64 ? sizeof(double) : sizeof(float)));
}

int rrtb_render_group(rrtb_ctx *const *ctxs, int n, const rrtb_render_params *p, int frame_f64, void *out_rgb, rrtb_stats *stats)
{
    if (!ctxs || n < 1 || !p || !out_rgb) return RRTB_ERR_INVALID;
    for (int i = 0; i < n; ++i)
        if (!ctxs[i]) return RRTB_ERR_INVALID;
    rrtb_ctx *owner = ctxs[0];
    int rc;
    if (!owner->d_frame || owner->peer_frame || owner->frame_w != p->width || owner->frame_h != p->height ||
        owner->frame_f64 != (frame_f64 ? 1 : 0)) {
        if ((rc = rrtb_frame_create(owner, p->width, p->height, frame_f64))) return rc;
        for (int i = 1; i < n; ++i) frame_drop_mapping(ctxs[i]);
    }
    for (int i = 1; i < n; ++i)
        if (ctxs[i]->peer_frame != owner->d_frame && (rc = rrtb_frame_attach(ctxs[i], owner))) {
            owner->err = ctxs[i]->err;
            return rc;
        }
    // every device gets its whole shard enqueued before anybody waits: the GPUs run concurrently from one host thread
    rrtb_render_params q = *p;
    q.world = n;
    for (int i = 0; i < n; ++i) {
        q.rank = i;
        if ((rc = enqueue_shard(ctxs[i], &q))) {
            owner->err = ctxs[i]->err;
            return rc;
        }
    }
    rrtb_stats total;
    memset(&total, 0, sizeof(total));
    for (int i = 0; i < n; ++i) {
        rrtb_stats st;
        if ((rc = finish_shard(ctxs[i], &st))) {
            owner->err = ctxs[i]->err;
            return rc;
        }
        total.seconds_render = st.seconds_render > total.seconds_render ? st.seconds_render : total.seconds_render;
        total.seconds_resolve = st.seconds_resolve > total.seconds_resolve ? st.seconds_resolve : total.seconds_resolve;
        total.seconds_build = st.seconds_build > total.seconds_build ? st.seconds_build : total.seconds_build;
        total.rays += st.rays; total.paths += st.paths; total.box_tests += st.box_tests; total.sphere_tests += st.sphere_tests;
        total.msphere_tests += st.msphere_tests; total.triangle_tests += st.triangle_tests; total.hits += st.hits;
        total.kernel_launches += st.kernel_launches;
    }
    if ((rc = rrtb_frame_download(owner, p->shard_mode, out_rgb))) return rc;
    if (stats) *stats = total;
    return RRTB_OK;
}

void *rrtb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void rrtb_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

int rrtb_probe_issue_rate(rrtb_ctx *ctx, double *ffma_lane_instr_per_s, double *mix_lane_instr_per_s)
{
    if (!ctx) return RRTB_ERR_INVALID;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if (ffma_lane_instr_per_s && (rc = launch_probe(ctx, 0, ffma_lane_instr_per_s))) return rc;
    if (mix_lane_instr_per_s && (rc = launch_probe(ctx, 1, mix_lane_instr_per_s))) return rc;
    return RRTB_OK;
}

} // extern "C"

// ---- test hooks: one body per hook, for the float (real = float) and the double integrator --------------------
namespace {
template <typename real>
int trace_hook(rrtb_ctx *ctx, const real *rays7, int n, real t_min, int mode, int32_t *id, real *t, real *rec7)
{
    if (!ctx || !rays7 || !id || !t || n < 0) return RRTB_ERR_INVALID;
    int rc;
    if ((rc = require_scene(ctx, "trace before rrtb_scene_set"))) return rc;
    if (!(t_min >= (real)0)) return invalid(ctx, "t_min must be >= 0 (the reference uses 0.001, rrt.cu:49)");
    if (n == 0) return RRTB_OK;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    DeviceArray<real> dr, dt, drec;
    DeviceArray<int32_t> di;
    if ((rc = dr.reserve(ctx, 7 * (size_t)n)) || (rc = di.reserve(ctx, n)) || (rc = dt.reserve(ctx, n)) ||
        (rec7 && (rc = drec.reserve(ctx, 7 * (size_t)n))))
        return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(dr, rays7, sizeof(real) * 7 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = launch_trace<real>(ctx, dr, n, t_min, mode ? 1 : 0, di, dt, drec))) return rc; // drec: null without rec7
    RRTB_CUDA(ctx, cudaMemcpyAsync(id, di, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    RRTB_CUDA(ctx, cudaMemcpyAsync(t, dt, sizeof(real) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (rec7) RRTB_CUDA(ctx, cudaMemcpyAsync(rec7, drec, sizeof(real) * 7 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

template <typename real>
int camera_rays_hook(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *pix, int n, int sample, real *rays7)
{
    if (!ctx || !p || !pix || !rays7 || n < 0) return RRTB_ERR_INVALID;
    int rc;
    if ((rc = require_scene(ctx, "camera rays before rrtb_scene_set"))) return rc;
    if (n == 0) return RRTB_OK;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    DeviceArray<int32_t> dp;
    DeviceArray<real> dr;
    if ((rc = dp.reserve(ctx, n)) || (rc = dr.reserve(ctx, 7 * (size_t)n))) return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(dp, pix, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = launch_camera_rays<real>(ctx, p, dp, n, sample, dr))) return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(rays7, dr, sizeof(real) * 7 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

template <typename real>
int scatter_hook(rrtb_ctx *ctx, const real *in16, const uint32_t *rnd4, int n, real *out8)
{
    if (!ctx || !in16 || !rnd4 || !out8 || n < 0) return RRTB_ERR_INVALID;
    int rc;
    if ((rc = require_scene(ctx, "scatter before rrtb_scene_set"))) return rc;
    if (n == 0) return RRTB_OK;
    for (int i = 0; i < n; ++i) { // the kernel indexes the material arrays with in16[14]
        const real m = in16[16 * (size_t)i + 14];
        if (!(m >= (real)0 && m < (real)ctx->n_materials)) return invalid(ctx, "scatter: material index out of range");
    }
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    DeviceArray<real> di, dout;
    DeviceArray<uint32_t> dr;
    if ((rc = di.reserve(ctx, 16 * (size_t)n)) || (rc = dr.reserve(ctx, 4 * (size_t)n)) || (rc = dout.reserve(ctx, 8 * (size_t)n)))
        return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(di, in16, sizeof(real) * 16 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    RRTB_CUDA(ctx, cudaMemcpyAsync(dr, rnd4, 16 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = launch_scatter<real>(ctx, di, dr, n, dout))) return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(out8, dout, sizeof(real) * 8 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}
} // namespace

extern "C" {

int rrtb_trace_closest(rrtb_ctx *ctx, const float *rays7, int n, float t_min, int mode, int32_t *id, float *t,
                       float *rec7)
{
    return trace_hook(ctx, rays7, n, t_min, mode, id, t, rec7);
}

int rrtb_trace_closest_f64(rrtb_ctx *ctx, const double *rays7, int n, double t_min, int mode, int32_t *id, double *t,
                           double *rec7)
{
    return trace_hook(ctx, rays7, n, t_min, mode, id, t, rec7);
}

int rrtb_camera_rays(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *pix, int n, int sample, float *rays7)
{
    return camera_rays_hook(ctx, p, pix, n, sample, rays7);
}

int rrtb_camera_rays_f64(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *pix, int n, int sample, double *rays7)
{
    return camera_rays_hook(ctx, p, pix, n, sample, rays7);
}

int rrtb_scatter(rrtb_ctx *ctx, const float *in16, const uint32_t *rnd4, int n, float *out8)
{
    return scatter_hook(ctx, in16, rnd4, n, out8);
}

int rrtb_scatter_f64(rrtb_ctx *ctx, const double *in16, const uint32_t *rnd4, int n, double *out8)
{
    return scatter_hook(ctx, in16, rnd4, n, out8);
}

int rrtb_bvh_size(rrtb_ctx *ctx, int32_t *n_prims)
{
    if (!ctx || !n_prims) return RRTB_ERR_INVALID;
    if (!ctx->has_scene) return RRTB_ERR_NO_SCENE;
    *n_prims = ctx->n_prims;
    return RRTB_OK;
}

int rrtb_bvh_download(rrtb_ctx *ctx, uint32_t *morton, uint32_t *perm, int32_t *left, int32_t *right,
                      int32_t *parent, float *node_box, float *prim_box)
{
    if (!ctx) return RRTB_ERR_INVALID;
    if (!ctx->has_scene) return RRTB_ERR_NO_SCENE;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->n_prims, ni = n > 0 ? n - 1 : 0;
    int rc;
    if (morton && (rc = read_back(ctx, morton, ctx->d_morton, 4 * n))) return rc;
    if (perm) {
        std::vector<uint64_t> keys(n);
        if ((rc = read_back(ctx, keys.data(), ctx->d_keys, 8 * n))) return rc;
        for (size_t k = 0; k < n; ++k) perm[k] = (uint32_t)keys[k];
    }
    if (left && ni && (rc = read_back(ctx, left, ctx->d_left, 4 * ni))) return rc;
    if (right && ni && (rc = read_back(ctx, right, ctx->d_right, 4 * ni))) return rc;
    if (parent && (rc = read_back(ctx, parent, ctx->d_parent, 4 * (2 * n - 1)))) return rc;
    if (node_box && ni) {
        if ((rc = refit_canonical(ctx)) || (rc = read_back(ctx, node_box, ctx->d_node_box, 4 * 6 * ni))) return rc;
    }
    if (prim_box && (rc = read_back(ctx, prim_box, ctx->d_prim_box, 4 * 6 * n))) return rc;
    return RRTB_OK;
}

int rrtb_wide_size(rrtb_ctx *ctx, int32_t *n_nodes, int32_t *width)
{
    if (!ctx || !n_nodes) return RRTB_ERR_INVALID;
    if (width) *width = RRTB_WIDTH;
    if (!ctx->has_scene) return RRTB_ERR_NO_SCENE;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    return read_back(ctx, n_nodes, ctx->d_collapse, sizeof(int)); // CollapseState::n_alloc
}

// IEEE half precision -> float (the half extents of the traversal nodes, rrtb_device.cuh "Traversal node")
static float f16_to_float(uint16_t h)
{
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16, e = (h >> 10) & 31u, m = h & 1023u;
    uint32_t b;
    if (e == 31u) b = sign | 0x7f800000u | (m << 13);            // inf / nan
    else if (e != 0u) b = sign | ((e + 112u) << 23) | (m << 13); // normal
    else if (m == 0u) b = sign;                                  // zero
    else {                                                       // subnormal: m * 2^-24
        float x = (float)m * 5.9604644775390625e-08f;
        memcpy(&b, &x, 4);
        b |= sign;
    }
    float x;
    memcpy(&x, &b, 4);
    return x;
}

int rrtb_wide_download(rrtb_ctx *ctx, float *nodes, int32_t max_nodes)
{
    if (!ctx || !nodes || max_nodes < 0) return RRTB_ERR_INVALID;
    int32_t n_nodes = 0;
    int rc = rrtb_wide_size(ctx, &n_nodes, nullptr);
    if (rc) return rc;
    if (n_nodes > max_nodes) return invalid(ctx, "wide-node buffer too small");
    // device nodes are 24 words with fp16 half extents (rrtb_device.cuh "Traversal node"), or 40 words with the boxes at
    // both ends of the shutter ("Motion node"); hand them back decoded, the motion node as the UNION of its two boxes
    const int words = ctx->motion ? 40 : 24;
    std::vector<uint32_t> raw((size_t)words * n_nodes);
    if ((rc = read_back(ctx, raw.data(), ctx->d_wnodes, sizeof(uint32_t) * raw.size()))) return rc;
    auto f = [](uint32_t b) {
        float x;
        memcpy(&x, &b, 4);
        return x;
    };
    for (int32_t i = 0; i < n_nodes; ++i) {
        const uint32_t *w = raw.data() + (size_t)words * i;
        float *o = nodes + (size_t)32 * i;
        const int hbase = ctx->motion ? 24 : 12, rbase = ctx->motion ? 36 : 18;
        for (int axis = 0; axis < 3; ++axis)
            for (int c = 0; c < 4; ++c) {
                const int pw = 2 * axis + c / 2; // the pair word of (axis, child pair)
                auto half = [&](int base) { return f16_to_float((uint16_t)((c & 1) ? w[base + pw] >> 16 : w[base + pw] & 0xffffu)); };
                float c0 = f(w[4 * axis + c]), h0 = half(hbase);
                if (ctx->motion) {
                    const float c1 = f(w[12 + 4 * axis + c]), h1 = half(hbase + 6);
                    const float lo = fminf(c0 - h0, c1 - h1), hi = fmaxf(c0 + h0, c1 + h1);
                    if (h0 == -INFINITY) h0 = -INFINITY; // unused slot stays unused
                    else {
                        c0 = 0.5f * (lo + hi);
                        h0 = fmaxf(hi - c0, c0 - lo);
                    }
                }
                o[4 * axis + c] = c0;
                o[12 + 4 * axis + c] = h0;
            }
        for (int k = 0; k < 4; ++k) memcpy(&o[24 + k], &w[rbase + k], 4);
        for (int k = 0; k < 4; ++k) o[28 + k] = 0.f;
    }
    return RRTB_OK;
}

int rrtb_wide_download_raw(rrtb_ctx *ctx, uint32_t *words, int32_t max_nodes, int32_t *words_per_node)
{
    if (!ctx || !words || max_nodes < 0) return RRTB_ERR_INVALID;
    int32_t n_nodes = 0;
    int rc = rrtb_wide_size(ctx, &n_nodes, nullptr);
    if (rc) return rc;
    if (n_nodes > max_nodes) return invalid(ctx, "wide-node buffer too small");
    const int wpn = ctx->motion ? 4 * RRTB_MOTION_NODE_F4 : 4 * RRTB_NODE_F4;
    if (words_per_node) *words_per_node = wpn;
    return read_back(ctx, words, ctx->d_wnodes, sizeof(uint32_t) * (size_t)wpn * n_nodes);
}

int rrtb_philox(rrtb_ctx *ctx, const uint32_t *ctr4, int n, uint32_t key0, uint32_t key1, uint32_t *out4)
{
    if (!ctx || !ctr4 || !out4 || n < 0) return RRTB_ERR_INVALID;
    if (n == 0) return RRTB_OK;
    RRTB_CUDA(ctx, cudaSetDevice(ctx->device));
    DeviceArray<uint32_t> dc, dout;
    int rc;
    if ((rc = dc.reserve(ctx, 4 * (size_t)n)) || (rc = dout.reserve(ctx, 4 * (size_t)n))) return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(dc, ctr4, 16 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = launch_philox(ctx, dc, n, key0, key1, dout))) return rc;
    RRTB_CUDA(ctx, cudaMemcpyAsync(out4, dout, 16 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    RRTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RRTB_OK;
}

} // extern "C"
