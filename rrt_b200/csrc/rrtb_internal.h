// rrtb_internal.h -- host-side context shared by the translation units of librrtb200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/rrtb.h"
#include "rrtb_device.cuh"

namespace rrtb {

// error helper: records the reference-style message (rrt.cu:31-40) and returns RRTB_ERR_CUDA
int cuda_fail(rrtb_ctx *ctx, cudaError_t e, const char *expr, const char *file, int line);

#define RRTB_CUDA(ctx, expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) return ::rrtb::cuda_fail((ctx), _e, #expr, __FILE__, __LINE__); \
    } while (0)

// One owning allocation of Ts: device memory (cudaMalloc), or pinned host memory (cudaHostAlloc) when PINNED.  Grow-only:
// reserve() reallocates, without keeping the contents, only when the request exceeds the count already held, so a frame
// loop that re-sends its scene pays no cudaMalloc / cudaFree.  Converts to T* for kernel arguments and pointer
// arithmetic; get() for a cast to another pointer type.
template <typename T, bool PINNED>
class CudaArray {
  public:
    CudaArray() = default;
    CudaArray(const CudaArray &) = delete;
    CudaArray &operator=(const CudaArray &) = delete;
    ~CudaArray() { release(); }
    operator T *() const { return p_; }
    T *get() const { return p_; }

    int reserve(rrtb_ctx *ctx, size_t count)
    {
        if (count == 0) count = 1;
        if (count <= cap_) return RRTB_OK;
        release();
        void *p = nullptr;
        RRTB_CUDA(ctx, PINNED ? cudaHostAlloc(&p, count * sizeof(T), cudaHostAllocPortable) : cudaMalloc(&p, count * sizeof(T)));
        p_ = (T *)p;
        cap_ = count;
        return RRTB_OK;
    }

  private:
    void release()
    {
        if (p_ && PINNED) cudaFreeHost(p_);
        else if (p_) cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    T *p_ = nullptr;
    size_t cap_ = 0;
};
template <typename T> using DeviceArray = CudaArray<T, false>;
template <typename T> using PinnedArray = CudaArray<T, true>;

} // namespace rrtb

// A new per-context buffer is one DeviceArray member: it is reserved where it is used and freed with the context.
struct rrtb_ctx {
    template <typename T> using DeviceArray = rrtb::DeviceArray<T>;
    template <typename T> using PinnedArray = rrtb::PinnedArray<T>;

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
    DeviceArray<float4> d_prim;       // [3*n] leaf records in object-id order (== flat_leaves)
    DeviceArray<int2> d_prim_info;    // [n]   (object id, material)
    DeviceArray<float4> d_materials;  // [nm]
    DeviceArray<int> d_material_type; // [nm]
    // device: canonical LBVH arrays (rrtb_bvh_download)
    DeviceArray<float> d_prim_box;    // [6n]
    DeviceArray<uint32_t> d_morton;   // [n]
    DeviceArray<uint64_t> d_keys;     // [n] sorted (code << 32 | id)
    DeviceArray<uint64_t> d_keys_tmp; // [n]
    DeviceArray<int> d_left, d_right; // [n-1]
    DeviceArray<int> d_parent;        // [2n-1]
    DeviceArray<float> d_node_box;    // [6(n-1)]
    bool canonical_boxes = false;     // d_node_box holds the refit of the canonical tree (else: refit_canonical on demand)
    // scenes with motion (moving primitives and an open shutter): boxes at the two ends of the shutter, for the
    // interpolating traversal nodes (rrtb_device.cuh "Motion node")
    bool motion = false;
    DeviceArray<float> d_prim_box01;  // [12n]
    DeviceArray<float> d_node_box01;  // [12(n-1)]
    DeviceArray<int> d_visit;         // [n-1]
    // SAH-rebuilt copy of the topology, for the traversal tree only (rrtb_bvh.cu k_sah_rebuild)
    DeviceArray<int2> d_range;        // [n-1] sorted positions covered by each canonical internal node
    DeviceArray<int> d_left2, d_right2; // [n-1]
    DeviceArray<int> d_parent2;       // [2n-1]
    DeviceArray<float> d_node_box2;   // [6(n-1)]
    DeviceArray<int> d_sah_roots;     // [n] roots of the subtrees to rebuild
    // device: traversal structures
    DeviceArray<float4> d_wnodes;     // [8*max(n-1,1)] 4-wide traversal nodes (rrtb_bvh.cu k_collapse4)
    DeviceArray<int> d_wq;            // [n] collapse work list: binary node that roots wide node i
    DeviceArray<int> d_collapse;      // CollapseState (wide-node count, ticket, leaves emitted)
    DeviceArray<float4> d_leaves;     // [3n] leaf order
    DeviceArray<int2> d_leaf_info;    // [n]
    DeviceArray<float4> d_prim_ext;   // [2n] edge rates of moving triangles, object-id order (allocated when the scene has any)
    DeviceArray<float4> d_leaf_ext;   // [2n] the same in leaf order
    // scratch
    DeviceArray<float> d_reduce;      // block partials + build constants
    DeviceArray<unsigned int> d_hist; // radix histograms
    DeviceArray<unsigned long long> d_counters; // [0] work queue head, [1] ray counter
    DeviceArray<uint64_t> d_accum;    // host-path accumulator (3*W*H)
    DeviceArray<double> d_rgb;        // host-path framebuffer, 3*W*H doubles' worth of room (float or double resolve)
    DeviceArray<float> d_aov;         // rrtb_render_aov's output, 8*W*H floats
    DeviceArray<unsigned char> d_stage; // raw scene structs of the last upload (input of k_prepare; kept for rebuilds)
    size_t stage_off[4] = {0, 0, 0, 0}; // byte offsets of the sphere / msphere / triangle / mtriangle arrays in d_stage
    float build_cam_mag = 0.f;        // camera magnitude the traversal-box padding was computed with
    rrtb_render_params pending{};     // the render enqueued by launch_render, for finish_render
    int pending_launches = 0;
    // multi-GPU frame (SURVEY 8e): the owner (rank 0) holds the float/double frame every rank's resolve epilogue stores its
    // tiles into, and the 64-bit sum buffer sample shards add into; other ranks hold peer mappings of both.  The two are
    // cudaMalloc'ed one each (not sub-allocated): CUDA IPC exports them.
    DeviceArray<double> d_frame;      // owner: 3*W*H doubles' worth of room (float or double frame)
    DeviceArray<uint64_t> d_sum;      // owner: 3*W*H fixed-point sums of a sample-sharded frame
    int frame_w = 0, frame_h = 0, frame_f64 = 0;
    void *peer_frame = nullptr;       // non-owner: the owner's d_frame / d_sum (IPC mapping or same-process pointer)
    uint64_t *peer_sum = nullptr;
    bool peer_is_ipc = false;
    PinnedArray<unsigned char> h_pinned; // staging for device->host copies into pageable user buffers
    PinnedArray<int> h_state;         // CollapseState read back behind every build

    ~rrtb_ctx(); // closes the peer mappings, destroys the events and the stream; the arrays free themselves
};

namespace rrtb {

// rrtb_api.cu
// device -> host copy on the context's stream, behind the kernels that wrote d_src; synchronises
int read_back(rrtb_ctx *ctx, void *dst, const void *d_src, size_t bytes);

// rrtb_bvh.cu
int prepare_and_build(rrtb_ctx *ctx); // from the raw scene in d_stage
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
