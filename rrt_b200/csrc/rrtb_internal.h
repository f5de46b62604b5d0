// rrtb_internal.h -- host-side context shared by the translation units of librrtb200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/rrtb.h"
#include "rrtb_device.cuh"

struct rrtb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr, ev_copy[2] = {nullptr, nullptr};
    int sm_count = 0;
    std::string err;

    // scene (host copies kept for camera updates / introspection)
    bool has_scene = false;
    rrtb_camera cam{};
    int n_materials = 0, n_spheres = 0, n_mspheres = 0, n_triangles = 0, n_mtriangles = 0, n_prims = 0;
    std::vector<rrtb_mtriangle> staged_mtriangles; // rrtb_scene_stage_moving_triangles -> next rrtb_scene_set
    bool staged_background = false;                // rrtb_scene_stage_background -> next rrtb_scene_set
    float staged_bg[3] = {0.f, 0.f, 0.f};
    bool background = false;                       // the loaded scene has a constant background bg instead of the sky
    float bg[3] = {0.f, 0.f, 0.f};
    bool lights = false;                           // ... or a RRTB_DIFFUSE_LIGHT material: render with the LIGHTS kernels
    int use_bvh = 1;
    double seconds_build = 0.0;

    // device: canonical primitive arrays (object-id order)
    float4 *d_prim = nullptr;       // [3*n] leaf records in object-id order (== flat_leaves)
    int2 *d_prim_info = nullptr;    // [n]   (object id, material)
    float4 *d_materials = nullptr;  // [nm]
    int *d_material_type = nullptr; // [nm]
    // device: canonical LBVH arrays (rrtb_bvh_download)
    float *d_prim_box = nullptr;    // [6n]
    uint32_t *d_morton = nullptr;   // [n]
    uint64_t *d_keys = nullptr;     // [n] sorted (code << 32 | id)
    uint64_t *d_keys_tmp = nullptr; // [n]
    int *d_left = nullptr, *d_right = nullptr; // [n-1]
    int *d_parent = nullptr;        // [2n-1]
    float *d_node_box = nullptr;    // [6(n-1)]
    bool canonical_boxes = false;   // d_node_box holds the refit of the canonical tree (else: refit_canonical on demand)
    // scenes with motion (moving primitives and an open shutter): boxes at the two ends of the shutter, for the
    // interpolating traversal nodes (rrtb_device.cuh "Motion node")
    bool motion = false;
    float *d_prim_box01 = nullptr;  // [12n]
    float *d_node_box01 = nullptr;  // [12(n-1)]
    int *d_visit = nullptr;         // [n-1]
    // SAH-rebuilt copy of the topology, for the traversal tree only (rrtb_bvh.cu k_sah_rebuild)
    int2 *d_range = nullptr;        // [n-1] sorted positions covered by each canonical internal node
    int *d_left2 = nullptr, *d_right2 = nullptr; // [n-1]
    int *d_parent2 = nullptr;       // [2n-1]
    float *d_node_box2 = nullptr;   // [6(n-1)]
    int *d_sah_roots = nullptr;     // [n] roots of the subtrees to rebuild
    // device: traversal structures
    float4 *d_wnodes = nullptr;     // [8*max(n-1,1)] 4-wide traversal nodes (rrtb_bvh.cu k_collapse4)
    int *d_wq = nullptr;            // [n] collapse work list: binary node that roots wide node i
    int *d_collapse = nullptr;      // CollapseState (wide-node count, ticket, leaves emitted)
    float4 *d_leaves = nullptr;     // [3n] leaf order
    int2 *d_leaf_info = nullptr;    // [n]
    float4 *d_prim_ext = nullptr;   // [2n] edge rates of moving triangles, object-id order (allocated when the scene has any)
    float4 *d_leaf_ext = nullptr;   // [2n] the same in leaf order
    // scratch
    float *d_reduce = nullptr;      // block partials + build constants
    unsigned int *d_hist = nullptr; // radix histograms
    size_t hist_elems = 0;
    unsigned long long *d_counters = nullptr; // [0] work queue head, [1] ray counter
    unsigned long long *d_accum = nullptr;    // host-path accumulator (3*W*H)
    float *d_rgb = nullptr;                   // host-path float framebuffer
    size_t accum_elems = 0;
    float *d_aov = nullptr;                   // rrtb_render_aov's output, 8*W*H floats (grow-only)
    unsigned char *d_stage = nullptr;         // raw scene structs of the last upload (input of k_prepare; kept for rebuilds)
    size_t stage_off[4] = {0, 0, 0, 0};       // byte offsets of the sphere / msphere / triangle / mtriangle arrays in d_stage
    float build_cam_mag = 0.f;                // camera magnitude the traversal-box padding was computed with
    rrtb_render_params pending{};             // the render enqueued by launch_render, for finish_render
    int pending_launches = 0;
    // multi-GPU frame (SURVEY 8e): the owner (rank 0) holds the float/double frame every rank's resolve epilogue stores its
    // tiles into, and the 64-bit sum buffer sample shards add into; other ranks hold peer mappings of both
    void *d_frame = nullptr;                  // owner: 3*W*H doubles' worth of room (float or double frame)
    unsigned long long *d_sum = nullptr;      // owner: 3*W*H fixed-point sums of a sample-sharded frame
    size_t frame_elems = 0;                   // 3*W*H the frame was sized for
    int frame_w = 0, frame_h = 0, frame_f64 = 0;
    void *peer_frame = nullptr;               // non-owner: the owner's d_frame / d_sum (IPC mapping or same-process pointer)
    unsigned long long *peer_sum = nullptr;
    bool peer_is_ipc = false;
    void *h_pinned = nullptr;                 // pinned staging for device->host copies into pageable user buffers
    size_t h_pinned_bytes = 0;
    int *h_state = nullptr;                   // pinned: CollapseState read back behind every build
    // Device buffers are grow-only: rrtb_scene_set re-uses them when the next scene fits (a frame loop that re-sends
    // its scene pays no cudaMalloc / cudaFree).  Capacity in bytes, keyed by the address of the pointer member.
    std::unordered_map<const void *, size_t> capacity;
};

namespace rrtb {

// error helper: records the reference-style message (rrt.cu:31-40) and returns RRTB_ERR_CUDA
int cuda_fail(rrtb_ctx *ctx, cudaError_t e, const char *expr, const char *file, int line);

#define RRTB_CUDA(ctx, expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) return ::rrtb::cuda_fail((ctx), _e, #expr, __FILE__, __LINE__); \
    } while (0)

// rrtb_bvh.cu
void free_scene(rrtb_ctx *ctx);
int refit_canonical(rrtb_ctx *ctx);

// rrtb_render.cu
DeviceScene device_scene(const rrtb_ctx *ctx);
DeviceCamera device_camera(const rrtb_camera &c, int W, int H);
int launch_render(rrtb_ctx *ctx, const rrtb_render_params *p, uint64_t *d_accum, rrtb_stats *stats, bool defer = false);
int finish_render(rrtb_ctx *ctx, rrtb_stats *stats);
// first-hit AOVs of a tile shard into d_out (8*W*H floats, planar: albedo, normal, depth, coverage); synchronises
int launch_aov(rrtb_ctx *ctx, const rrtb_render_params *p, float *d_out, rrtb_stats *stats);
int launch_resolve_tiles(rrtb_ctx *ctx, const uint64_t *d_accum, void *d_out, const rrtb_render_params *p, bool f64);
int launch_accumulate_atomic(rrtb_ctx *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t n);
int launch_accumulate(rrtb_ctx *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t n);
int launch_philox(rrtb_ctx *ctx, const uint32_t *d_ctr, int n, uint32_t k0, uint32_t k1, uint32_t *d_out);
int launch_probe(rrtb_ctx *ctx, int mix, double *lane_instr_per_s);
// T / real = float: the float integrator and framebuffer, double: the double ones (instantiated for both)
template <typename T>
int launch_resolve(rrtb_ctx *ctx, const uint64_t *d_accum, T *d_out, size_t n);
template <typename real>
int launch_trace(rrtb_ctx *ctx, const real *d_rays7, int n, real t_min, int mode, int32_t *d_id, real *d_t, real *d_rec7);
template <typename real>
int launch_camera_rays(rrtb_ctx *ctx, const rrtb_render_params *p, const int32_t *d_pix, int n, int sample, real *d_rays7);
template <typename real>
int launch_scatter(rrtb_ctx *ctx, const real *d_in16, const uint32_t *d_rnd4, int n, real *d_out8);

} // namespace rrtb
