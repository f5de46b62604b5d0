// rrtb_render_pool.cuh -- scheduler RRTB_SCHED_POOL: a per-warp on-chip wavefront (sm_100a).
//
// Why (ncu, profiles/README.md): with one path per lane a warp runs at 7-12 of 32 lanes -- every lane
// waits for the slowest traversal of the round (node visits per ray: mean 12, tail > 60) and the shading
// code runs once per round whatever the number of lanes that need it.
//
// Here each WARP owns a pool of POOL path slots in shared memory (60 B per slot; 228 KB/SM makes room for
// 24 warps x 128 slots) and runs a small warp-synchronous scheduler over three stacks of slot ids:
//
//   trace stack    slots whose ray awaits traversal
//   scatter stack  slots whose segment HIT something  (hit record + material scatter next)
//   gen stack      slots whose path ENDED (sky, absorbed, depth, emitter) or that never held one
//
//   FETCH    idle lanes pop the trace stack, load the ray and start a traversal
//   STEP     lanes in flight visit BVH nodes (the inner loop runs on while a vote finds enough of them),
//            then, by vote, do one exact leaf test; a lane whose traversal ends writes (t, leaf ref) to its
//            slot, pushes it on the scatter or the gen stack and is idle at once -- nobody waits for it
//   SCATTER  32 hit slots, one per lane: hit record, Philox block, scatter; survivors -> trace stack (LIGHTS: an
//            emitter hit adds throughput x Le to the accumulator here and ends its path)
//   GEN      32 ended slots, one per lane: sky (LIGHTS: or background) x throughput into the accumulator (64-bit integer atomics),
//            then the next camera paths of the global queue (ONE warp-aggregated atomicAdd per batch),
//            Philox block, thin-lens ray -> trace stack
//
// SCATTER and GEN are separate batches so that each runs its own straight-line code 32 lanes wide (as one
// batch the hit/miss branches serialised at ~15 lanes).  Lanes in the middle of a traversal keep their
// traversal registers across a batch and resume.  Nothing but the per-path radiance leaves the SM.
// Everything is keyed by (pixel, sample, bounce), so the image is bit-identical to the other schedulers.
//
// The kernel is written once over the path policy of rrtb_path.cuh: PathF32 is the float integrator (the headline
// build, 64 registers, 4 blocks/SM, 60-byte slots), PathF64 the double integrator (SURVEY 8f1: double ray /
// throughput / hit distance in the slot, 107-byte slots, 3 blocks/SM).
#pragma once
#include "rrtb_path.cuh"

namespace rrtb {

static constexpr int POOL_WARPS = RENDER_TPB / 32;
static constexpr int SLOT_FRESH = -2;          // hit_ref marker: nothing to accumulate for this slot

template <typename real, int POOL>
struct WarpPoolT { // SoA, one per warp, in dynamic shared memory
    real ox[POOL], oy[POOL], oz[POOL], dx[POOL], dy[POOL], dz[POOL], tm[POOL];
    real tr[POOL], tg[POOL], tb[POOL];
    real hit_t[POOL];
    int pixel[POOL], sample[POOL], bounce[POOL];
    int hit_ref[POOL];
    unsigned char tq[POOL]; // trace stack
    unsigned char sq[POOL]; // scatter stack
    unsigned char gq[POOL]; // gen stack
};

// LIGHTS: the scene has emitters (RRTB_DIFFUSE_LIGHT) or a background; the other instantiations compile neither in
template <bool COUNT_RAYS, int NODE_UNROLL, bool MTRI = false, class P = PathF32, bool MOTION = false, bool LIGHTS = false>
__global__ void __launch_bounds__(RENDER_TPB, P::BLOCKS_PER_SM) k_render_pool(const RenderArgs a)
{
    typedef typename P::real real;
    typedef WarpPoolT<real, P::POOL> WarpPool;
    constexpr int POOL = P::POOL;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpPool &wp = reinterpret_cast<WarpPool *>(smem_raw)[threadIdx.x >> 5];
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const DeviceScene &s = a.scene;
    const float4 *__restrict__ wnodes = s.wnodes;
    const float4 *__restrict__ leaves = s.leaves;
    const LeafAux info = {s.leaf_info, s.leaf_ext};
    const real t_min = (real)0.001; // rrt.cu:49

    // every slot starts on the gen stack with nothing to accumulate
    for (int k = lane; k < POOL; k += 32) {
        wp.gq[k] = (unsigned char)k;
        wp.hit_ref[k] = SLOT_FRESH;
    }
    __syncwarp();
    // stack heights are warp-uniform and live in registers: every lane derives them from the same ballots
    int tq_n = 0, sq_n = 0, gq_n = POOL;

    // lane state: the traversal in flight (slot < 0: idle, and then cur == TRAV_DONE)
    int slot = -1;
    typename P::RayT ray;
    RayPre pre;
    int cur = TRAV_DONE;
    int stack[RRTB_STACK];
    TravSp sp = TravSp();
    typename P::HitT best = P::make_hit((real)0, -1);
    bool queue_empty = false; // the global work queue has run dry (warp-uniform)
    unsigned long long rays = 0, hits = 0;
    TravCounters tc = {0ull, 0ull, 0ull, 0ull};

    while (true) {
        const unsigned idle_mask = __ballot_sync(0xffffffffu, slot < 0);
        const int n_idle = __popc(idle_mask);
        // partial batches only when the trace stack is dry and enough lanes have nothing to do
        const bool starving = tq_n == 0 && n_idle >= a.th_shade;

        if (n_idle >= a.th_fetch && tq_n > 0) {
            // ---------------- FETCH: idle lanes pop slots off the trace stack
            const int take = min(n_idle, tq_n);
            const int rank = __popc(idle_mask & lt_mask);
            if (slot < 0 && rank < take) {
                slot = wp.tq[tq_n - 1 - rank];
                RRTB_CHECK(slot >= 0 && slot < POOL && tq_n - 1 - rank >= 0);
                ray.ox = wp.ox[slot]; ray.oy = wp.oy[slot]; ray.oz = wp.oz[slot];
                ray.dx = wp.dx[slot]; ray.dy = wp.dy[slot]; ray.dz = wp.dz[slot];
                ray.tm = wp.tm[slot];
                pre = P::pre(ray);
                if (MOTION) pre.s = ((float)ray.tm - s.shutter_open) * s.shutter_inv; // where the ray's time lies in the shutter
                best.t = P::inf();
                best.ref = -1;
                trav_begin(cur, sp, stack);
            }
            tq_n -= take;
        }
        else if (sq_n >= 32 || (starving && sq_n > 0 && sq_n >= gq_n)) {
            // ---------------- SCATTER: up to 32 hit slots, one per lane (rrt.cu:50-60)
            const int take = min(32, sq_n);
            const bool mine = (int)lane < take;
            const int sl = mine ? wp.sq[sq_n - 1 - lane] : 0;
            sq_n -= take;
            __syncwarp(); // every lane has read its slot id before the stacks are pushed to below
            bool to_trace = false, ended = false;
            if (mine) {
                typename P::RayT r;
                r.ox = wp.ox[sl]; r.oy = wp.oy[sl]; r.oz = wp.oz[sl];
                r.dx = wp.dx[sl]; r.dy = wp.dy[sl]; r.dz = wp.dz[sl];
                r.tm = wp.tm[sl];
                const int bounce = wp.bounce[sl];
                const typename P::HitT h = P::make_hit(wp.hit_t[sl], wp.hit_ref[sl]);
                if (COUNT_RAYS) {
                    ++rays;
                    ++hits;
                }
                typename P::RecT rec = P::template record<MTRI>(leaves, info, r, h);
                uint4 rnd = philox4x32_10(make_uint4((uint32_t)wp.pixel[sl], (uint32_t)wp.sample[sl], 2u + (uint32_t)bounce, 0u), a.key);
                float4 m = __ldg(&s.materials[rec.mat]);
                int mtype = __ldg(&s.material_type[rec.mat]);
                real dx, dy, dz, ar, ag, ab;
                if (P::template bounce<LIGHTS>(mtype, m, r, rec, rnd, dx, dy, dz, ar, ag, ab) && bounce + 1 < a.max_depth) {
                    wp.ox[sl] = rec.px; wp.oy[sl] = rec.py; wp.oz[sl] = rec.pz;
                    wp.dx[sl] = dx; wp.dy[sl] = dy; wp.dz[sl] = dz;
                    wp.tr[sl] = P::mul(wp.tr[sl], ar); wp.tg[sl] = P::mul(wp.tg[sl], ag); wp.tb[sl] = P::mul(wp.tb[sl], ab);
                    wp.bounce[sl] = bounce + 1;
                    to_trace = true;
                }
                else { // absorbed (rrt.cu:61-63) or depth exhausted (rrt.cu:78): black, nothing to accumulate
                    if constexpr (LIGHTS) { // ... unless an emitter ended the path: throughput x Le, accumulated here
                        if (mtype == RRTB_DIFFUSE_LIGHT) {
                            unsigned long long fr, fg, fb;
                            P::const_fixed(wp.tr[sl], wp.tg[sl], wp.tb[sl], m.x, m.y, m.z, a.clamp, fr, fg, fb);
                            unsigned long long *dst = a.accum + 3ull * (unsigned long long)wp.pixel[sl];
                            atomicAdd(dst + 0, fr);
                            atomicAdd(dst + 1, fg);
                            atomicAdd(dst + 2, fb);
                        }
                    }
                    wp.hit_ref[sl] = SLOT_FRESH;
                    ended = true;
                }
            }
            const unsigned t_mask = __ballot_sync(0xffffffffu, to_trace);
            const unsigned e_mask = __ballot_sync(0xffffffffu, ended);
            if (to_trace) wp.tq[tq_n + __popc(t_mask & lt_mask)] = (unsigned char)sl;
            if (ended) wp.gq[gq_n + __popc(e_mask & lt_mask)] = (unsigned char)sl;
            tq_n += __popc(t_mask);
            gq_n += __popc(e_mask);
            RRTB_CHECK(tq_n <= POOL && gq_n <= POOL && sq_n >= 0);
            __syncwarp(); // slot contents + stack entries visible to the lanes that will pop them
        }
        else if (gq_n >= 32 || (starving && gq_n > 0)) {
            // ---------------- GEN: up to 32 ended slots, one per lane: accumulate, then regenerate
            const int take = min(32, gq_n);
            const bool mine = (int)lane < take;
            const int sl = mine ? wp.gq[gq_n - 1 - lane] : 0;
            gq_n -= take;
            __syncwarp();
            if (mine && wp.hit_ref[sl] == -1) { // the segment left the scene: sky x throughput (rrt.cu:68-75), or background
                if (COUNT_RAYS) ++rays;
                unsigned long long fr, fg, fb;
                if (LIGHTS && a.background) {
                    P::const_fixed(wp.tr[sl], wp.tg[sl], wp.tb[sl], a.bg[0], a.bg[1], a.bg[2], a.clamp, fr, fg, fb);
                }
                else {
                    typename P::RayT r;
                    r.dx = wp.dx[sl]; r.dy = wp.dy[sl]; r.dz = wp.dz[sl];
                    P::sky_fixed(r, wp.tr[sl], wp.tg[sl], wp.tb[sl], a.clamp, fr, fg, fb);
                }
                unsigned long long *dst = a.accum + 3ull * (unsigned long long)wp.pixel[sl];
                atomicAdd(dst + 0, fr);
                atomicAdd(dst + 1, fg);
                atomicAdd(dst + 2, fb);
            }
            // next camera paths: one warp-aggregated atomic on the global queue
            bool to_trace = false;
            if (!queue_empty) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(a.queue, (unsigned long long)take);
                base = __shfl_sync(0xffffffffu, base, 0);
                if (base + (unsigned long long)take >= a.n_items) queue_empty = true;
                // decode (local tile, local sample) of the first item once per warp (64-bit division); the
                // other lanes are at most one (tile, sample) group further on
                const unsigned long long ts0 = base >> 5;
                int ls0 = 0, ltile0 = 0;
                if (lane == 0) {
                    ltile0 = (int)(ts0 / (unsigned long long)a.n_local_samples);
                    ls0 = (int)(ts0 - (unsigned long long)ltile0 * (unsigned long long)a.n_local_samples);
                }
                ls0 = __shfl_sync(0xffffffffu, ls0, 0);
                ltile0 = __shfl_sync(0xffffffffu, ltile0, 0);
                const unsigned long long item = base + lane;
                if (mine && item < a.n_items) {
                    // item = (local_tile * n_local_samples + local_sample) * 32 + pixel_in_tile
                    const unsigned pit = (unsigned)(item & 31ull);
                    int ls = ls0 + (int)((item >> 5) - ts0), ltile = ltile0;
                    if (ls >= a.n_local_samples) {
                        ls -= a.n_local_samples;
                        ++ltile;
                    }
                    const int tile = a.shard_mode == RRTB_SHARD_TILES ? ltile * a.world + a.rank : ltile;
                    int ty = (int)__fdividef((float)tile, (float)a.tiles_x); // float estimate, off by <= 1 ...
                    int tx = tile - ty * a.tiles_x;
                    if (tx < 0) { // ... corrected exactly in integers
                        --ty;
                        tx += a.tiles_x;
                    }
                    else if (tx >= a.tiles_x) {
                        ++ty;
                        tx -= a.tiles_x;
                    }
                    const int i = tx * 8 + (int)(pit & 7u), j = ty * 4 + (int)(pit >> 3);
                    if (i < a.W && j < a.H) { // else: padding pixel of an edge tile, the slot asks again
                        const int sample = a.shard_mode == RRTB_SHARD_SAMPLES ? ls * a.world + a.rank : ls;
                        typename P::RayT r = P::camera(a.cam, a.W, a.H, i, j, sample, a.key); // rrt.cu:112-114, camera.h:31-38
                        wp.ox[sl] = r.ox; wp.oy[sl] = r.oy; wp.oz[sl] = r.oz;
                        wp.dx[sl] = r.dx; wp.dy[sl] = r.dy; wp.dz[sl] = r.dz;
                        wp.tm[sl] = r.tm;
                        wp.tr[sl] = (real)1; wp.tg[sl] = (real)1; wp.tb[sl] = (real)1;
                        RRTB_CHECK(sl >= 0 && sl < POOL && j * a.W + i < a.W * a.H);
                        wp.pixel[sl] = j * a.W + i;
                        wp.sample[sl] = sample;
                        wp.bounce[sl] = 0;
                        to_trace = true;
                    }
                }
            }
            // route: new ray -> trace stack; padding pixel -> gen stack again while the queue has work; else dead
            const bool again = mine && !to_trace && !queue_empty;
            if (mine && !to_trace) wp.hit_ref[sl] = SLOT_FRESH;
            const unsigned t_mask = __ballot_sync(0xffffffffu, to_trace);
            const unsigned g_mask = __ballot_sync(0xffffffffu, again);
            if (to_trace) wp.tq[tq_n + __popc(t_mask & lt_mask)] = (unsigned char)sl;
            if (again) wp.gq[gq_n + __popc(g_mask & lt_mask)] = (unsigned char)sl;
            tq_n += __popc(t_mask);
            gq_n += __popc(g_mask);
            RRTB_CHECK(tq_n <= POOL && gq_n <= POOL && tq_n + sq_n + gq_n <= POOL);
            __syncwarp();
        }
        else if (n_idle == 32) {
            break; // nothing in flight and all three stacks empty: every slot is dead
        }
        else {
            // ---------------- STEP: node visits continue while at least th_node lanes still have a node to
            // visit (one vote per visit, at most step_iters in a row), then, by vote, one exact leaf test
            int it = 0;
#pragma unroll 1
            do {
#pragma unroll
                for (int u = 0; u < NODE_UNROLL; ++u) // node visits between two continue-votes
                    if (cur >= 0) wide_step<COUNT_RAYS, MOTION>(wnodes, pre, P::t_min_f(t_min), P::t_max_f(best), cur, sp, stack, tc);
            } while (++it < a.step_iters && __popc(__ballot_sync(0xffffffffu, cur >= 0)) >= a.th_node);
            const bool at_leaf = cur < 0 && cur != TRAV_DONE;
            const unsigned leaf_mask = __ballot_sync(0xffffffffu, at_leaf);
            if (leaf_mask) {
                const unsigned node_mask = __ballot_sync(0xffffffffu, cur >= 0);
                if (__popc(leaf_mask) >= a.th_leaf || node_mask == 0u) {
                    if (at_leaf) leaf_step<P, COUNT_RAYS, MTRI>(leaves, info, ray, pre, t_min, best, cur, sp, stack, tc);
                }
            }
            // lanes whose traversal ended publish the hit and go idle
            const bool fin = slot >= 0 && cur == TRAV_DONE;
            const unsigned fin_mask = __ballot_sync(0xffffffffu, fin);
            if (fin_mask) {
                const bool hit = fin && best.ref >= 0;
                const unsigned hit_mask = __ballot_sync(0xffffffffu, hit);
                const unsigned miss_mask = fin_mask & ~hit_mask;
                if (fin) {
                    wp.hit_t[slot] = best.t;
                    wp.hit_ref[slot] = best.ref; // -1 = miss
                    if (hit) wp.sq[sq_n + __popc(hit_mask & lt_mask)] = (unsigned char)slot;
                    else wp.gq[gq_n + __popc(miss_mask & lt_mask)] = (unsigned char)slot;
                    slot = -1;
                }
                sq_n += __popc(hit_mask);
                gq_n += __popc(miss_mask);
                RRTB_CHECK(sq_n <= POOL && gq_n <= POOL && tq_n + sq_n + gq_n <= POOL);
                __syncwarp();
            }
        }
    }
    if (COUNT_RAYS) {
        unsigned long long v[6] = {rays, tc.box, tc.sph, tc.msph, tc.tri, hits};
        for (int k = 0; k < 6; ++k) {
            for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
            if (lane == 0 && v[k]) atomicAdd(a.queue + 1 + k, v[k]);
        }
    }
}

} // namespace rrtb
