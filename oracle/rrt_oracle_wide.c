/* rrt_oracle_wide.c -- TEST INFRASTRUCTURE ONLY: the traversal tree of the product, restated on the CPU.
 *
 * Starting from the canonical LBVH (orc_bvh_build), this file restates in float and in the GPU's operation order every
 * step of rrt_b200/csrc/rrtb_bvh.cu that turns the LBVH into the 4-wide tree the render kernels walk:
 *   k_sah_select     maximal subtrees of 3 .. SAH_MAX leaves under a node of more than SAH_MAX leaves
 *   k_sah_rebuild    binned SAH (32 bins on twice the centroid, lo + hi), prefix / exclusive-suffix unions, lowest
 *                    axis * 32 + bin on a tie, stable partition with the right side reversed; runs of 2..4 boxes by
 *                    exact enumeration of the splits (element 0 on the left, lowest mask on a tie); median split when
 *                    no plane has primitives on both sides or when the depth budget 63 - depth(root) runs out
 *   k_refit_upper    the Morton top above the subtrees, with its parent / grandparent rule for uncovered leaves
 *   k_prepare/k_refit<2>  the boxes at the two ends of the shutter (motion nodes)
 *   k_collapse4      greedy collapse (open the internal child of largest box_area6, first maximum wins) and the node
 *                    encoding: float centres, fp16 half extents rounded toward +inf, refs
 * Every product and sum is written as one C operation and the library is built with -ffp-contract=off, so each rounds
 * once, as the intrinsics of the CUDA side do.  Nodes come out in a CANONICAL order (pre-order from the root, children
 * in slot order); the GPU numbers them by atomics, which a test renumbers the same way before comparing words.
 */
#include "rrt_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define SAH_MAX 512
#define SAH_BINS 32
#define SAH_BIG 128
#define SMALL_SORT 2048
#define TRAV_DONE ((int32_t)0x80000000)

/* order-preserving float <-> int of the shared-memory bins (rrtb_bvh.cu f2o / o2f) */
static inline int32_t f2o(float f)
{
    int32_t b;
    memcpy(&b, &f, 4);
    return b >= 0 ? b : b ^ 0x7fffffff;
}
static inline float o2f(int32_t o)
{
    int32_t b = o >= 0 ? o : o ^ 0x7fffffff;
    float f;
    memcpy(&f, &b, 4);
    return f;
}

/* cvt.rzi.s32.f32: truncation toward zero, NaN -> 0, saturated to the int range */
static inline int f2i_rz(float x)
{
    if (x != x) return 0;
    if (x >= 2147483648.0f) return 0x7fffffff;
    if (x <= -2147483648.0f) return (int)0x80000000;
    return (int)x;
}

static inline int ceil_log2(int x) /* 32 - __clz(x - 1) for x >= 2 */
{
    int l = 0;
    while ((1u << l) < (unsigned)x) ++l;
    return l;
}

static inline int popc(unsigned x) { return __builtin_popcount(x); }

/* rrtb_bvh.cu area_rn, sah_cost_rn, centroid2, sah_scale, sah_bin: each product, sum and quotient rounds once */
static inline float area3(float x, float y, float z) { return x * y + y * z + z * x; }
static inline float box_area6(const float *b) { return area3(b[3] - b[0], b[4] - b[1], b[5] - b[2]); }
static inline float sah_cost(float a0, int n0, float a1, int n1) { return a0 * (float)n0 + a1 * (float)n1; }
static inline float centroid2(const float *b, int k) { return b[k] + b[3 + k]; }
static inline float sah_scale(float cmin, float cmax) { return cmax > cmin ? (float)SAH_BINS / (cmax - cmin) : 0.f; }
static inline int sah_bin(float c2, float cmin, float scale)
{
    const int j = f2i_rz((c2 - cmin) * scale);
    return j < SAH_BINS - 1 ? j : SAH_BINS - 1;
}

uint16_t orc_f16_up(float h)
{
    uint32_t u;
    memcpy(&u, &h, 4);
    const uint32_t sign = u >> 31, a = u & 0x7fffffffu;
    const uint16_t s16 = (uint16_t)(sign << 15);
    if (a > 0x7f800000u) return 0x7fff;            /* NaN */
    if (a == 0x7f800000u) return s16 | 0x7c00u;     /* +-inf */
    if (a == 0) return s16;                         /* +-0 */
    int e = (int)(a >> 23) - 127;
    uint64_t m = a & 0x7fffffu;
    if (a >> 23) m |= 0x800000u;
    else e = -126; /* float subnormal */
    /* |h| = m * 2^(e - 23); in units of the fp16 result's last place */
    uint64_t q, rem;
    uint32_t bits;
    if (e > 15) { /* beyond the fp16 range */
        return sign ? (uint16_t)(s16 | 0x7bffu) : (uint16_t)0x7c00u;
    }
    if (e >= -14) { /* fp16 normal: 10 fraction bits */
        q = m >> 13;
        rem = m & 0x1fffu;
        bits = (uint32_t)((e + 15) << 10) | (uint32_t)(q & 0x3ffu);
    }
    else { /* fp16 subnormal: units of 2^-24, |h| = m * 2^(e + 1) units */
        const int sh = -(e + 1);
        q = sh < 64 ? m >> sh : 0;
        rem = sh < 64 ? m & ((1ull << sh) - 1ull) : m;
        bits = (uint32_t)q;
    }
    if (!sign && rem) ++bits; /* toward +inf: a carry into the exponent is the next binade, or +inf */
    return (uint16_t)(s16 | bits);
}

static inline void center_half(float lo, float hi, float pad, float *c, float *h)
{
    *c = 0.5f * (lo + hi);
    const float a = hi - *c, b = *c - lo;
    *h = fmaxf(a, b) + pad;
}

static inline int prim_type(const orc_scene *s, int id)
{
    const int ns = s->n_spheres, nms = s->n_mspheres, nt = s->n_triangles;
    return id < ns ? 0 : (id < ns + nms ? 1 : (id < ns + nms + nt ? 2 : 3));
}

/* k_prepare prim_box01: lo/hi at camera time0, lo/hi at camera time1; a static primitive repeats its one box */
static void prim_box01(const orc_scene *s, int id, const float *box, float *o)
{
    const int ns = s->n_spheres, nms = s->n_mspheres, nt = s->n_triangles;
    const float t0 = s->cam.time0, t1 = s->cam.time1;
    if (id >= ns && id < ns + nms) {
        const rrtb_msphere *m = &s->mspheres[id - ns];
        const float dt = m->time1 - m->time0;
        const float k0 = (t0 - m->time0) / dt, k1 = (t1 - m->time0) / dt;
        const float ar = fabsf(m->radius);
        for (int k = 0; k < 3; ++k) {
            const float dc = m->center1[k] - m->center0[k];
            const float ca = m->center0[k] + k0 * dc, cb = m->center0[k] + k1 * dc;
            o[k] = ca - ar;
            o[3 + k] = ca + ar;
            o[6 + k] = cb - ar;
            o[9 + k] = cb + ar;
        }
    }
    else if (id >= ns + nms + nt) {
        float base[3], rate[3], e1b[3], e1r[3], e2b[3], e2r[3];
        orc_mtriangle_record2(&s->mtriangles[id - ns - nms - nt], base, rate, e1b, e1r, e2b, e2r);
        for (int k = 0; k < 3; ++k) {
            const float pa = fmaf(rate[k], t0, base[k]), pb = fmaf(rate[k], t1, base[k]);
            const float a1 = e1r[k] == 0.0f ? e1b[k] : fmaf(e1r[k], t0, e1b[k]), a2 = e2r[k] == 0.0f ? e2b[k] : fmaf(e2r[k], t0, e2b[k]);
            const float b1 = e1r[k] == 0.0f ? e1b[k] : fmaf(e1r[k], t1, e1b[k]), b2 = e2r[k] == 0.0f ? e2b[k] : fmaf(e2r[k], t1, e2b[k]);
            o[k] = fminf(fminf(pa, pa + a1), pa + a2);
            o[3 + k] = fmaxf(fmaxf(pa, pa + a1), pa + a2);
            o[6 + k] = fminf(fminf(pb, pb + b1), pb + b2);
            o[9 + k] = fmaxf(fmaxf(pb, pb + b1), pb + b2);
        }
    }
    else {
        memcpy(o, box, 6 * sizeof(float));
        memcpy(o + 6, box, 6 * sizeof(float));
    }
}

typedef struct builder {
    const orc_scene *s;
    const orc_bvh *b;
    int n, ni, nt_shape, motion;
    int32_t *left2, *right2, *parent2;
    float *node_box2, *node_box01, *pbox01;
    orc_wide *w;
    int cap_tasks, cap_items;
} builder;

static void log_task(builder *B, int path, const int *items, int cnt, int choice, int how, int level, int budget)
{
    orc_wide *w = B->w;
    if (w->n_tasks == B->cap_tasks) {
        B->cap_tasks = 2 * B->cap_tasks + 64;
        w->tasks = (int32_t *)realloc(w->tasks, sizeof(int32_t) * 7 * (size_t)B->cap_tasks);
    }
    if (w->n_items + cnt > B->cap_items) {
        B->cap_items = 2 * (B->cap_items + cnt) + 1024;
        w->items = (int32_t *)realloc(w->items, sizeof(int32_t) * (size_t)B->cap_items);
    }
    int32_t *t = w->tasks + 7 * (size_t)w->n_tasks++;
    t[0] = path;
    t[1] = w->n_items;
    t[2] = cnt;
    t[3] = choice;
    t[4] = how;
    t[5] = level;
    t[6] = budget;
    memcpy(w->items + w->n_items, items, sizeof(int) * (size_t)cnt);
    w->n_items += cnt;
}

typedef struct task {
    int node, cnt;
    int *items; /* sorted positions of the run, in run order */
} task;

/* one k_sah_rebuild task: choose, partition (items rewritten in place), return the left count and write the node box */
static int split_task(builder *B, int node, int *items, int cnt, int level, int budget)
{
    const float inf = INFINITY;
    const float *pb = B->b->prim_box;
    const uint32_t *perm = B->b->perm;
    orc_wide_counters *C = &B->w->cnt;
    float *nb = B->node_box2 + 6 * (size_t)node;
    int nl;
    if (cnt <= 4) {
        float lo4[4][3], hi4[4][3];
        for (int i = 0; i < cnt; ++i)
            for (int c = 0; c < 3; ++c) {
                lo4[i][c] = pb[6 * (size_t)perm[items[i]] + c];
                hi4[i][c] = pb[6 * (size_t)perm[items[i]] + 3 + c];
            }
        for (int c = 0; c < 3; ++c) {
            float lo = lo4[0][c], hi = hi4[0][c];
            for (int i = 1; i < cnt; ++i) {
                lo = fminf(lo, lo4[i][c]);
                hi = fmaxf(hi, hi4[i][c]);
            }
            nb[c] = lo;
            nb[3 + c] = hi;
        }
        float cost = inf;
        int best = 0;
        for (int lane = 0; lane < (1 << (cnt - 1)) - 1; ++lane) {
            const unsigned mask = 1u | ((unsigned)lane << 1);
            float alo[3] = {inf, inf, inf}, ahi[3] = {-inf, -inf, -inf}, blo[3] = {inf, inf, inf}, bhi[3] = {-inf, -inf, -inf};
            for (int i = 0; i < cnt; ++i)
                for (int c = 0; c < 3; ++c) {
                    if ((mask >> i) & 1u) {
                        alo[c] = fminf(alo[c], lo4[i][c]);
                        ahi[c] = fmaxf(ahi[c], hi4[i][c]);
                    }
                    else {
                        blo[c] = fminf(blo[c], lo4[i][c]);
                        bhi[c] = fmaxf(bhi[c], hi4[i][c]);
                    }
                }
            const int na = popc(mask & ((1u << cnt) - 1u));
            const float ck = sah_cost(area3(ahi[0] - alo[0], ahi[1] - alo[1], ahi[2] - alo[2]), na,
                                      area3(bhi[0] - blo[0], bhi[1] - blo[1], bhi[2] - blo[2]), cnt - na);
            if (ck < cost) { /* lanes in increasing order: the lowest lane wins a tie */
                cost = ck;
                best = lane;
            }
        }
        unsigned bm = 1u | ((unsigned)best << 1);
        int how = 0;
        if (!(cost < inf)) how = 1;
        else if (level + cnt - 1 >= budget) how = 2;
        if (how) bm = (1u << (cnt / 2)) - 1u;
        ++C->small_splits;
        if (how) ++C->small_halved;
        log_task(B, 2, items, cnt, (int)bm, how, level, budget);
        nl = popc(bm);
        int tmp[4], l = 0, r = nl;
        for (int i = 0; i < cnt; ++i) {
            if ((bm >> i) & 1u) tmp[l++] = items[i];
            else tmp[r++] = items[i];
        }
        memcpy(items, tmp, sizeof(int) * (size_t)cnt);
        return nl;
    }
    const int block = B->nt_shape >= SAH_MAX && cnt > SAH_BIG;
    /* centroid bounds, twice the centroid: lo + hi */
    float cmin[3] = {inf, inf, inf}, cmax[3] = {-inf, -inf, -inf}, scale[3];
    for (int i = 0; i < cnt; ++i) {
        const float *bx = pb + 6 * (size_t)perm[items[i]];
        for (int k = 0; k < 3; ++k) {
            const float c = centroid2(bx, k);
            cmin[k] = fminf(cmin[k], c);
            cmax[k] = fmaxf(cmax[k], c);
        }
    }
    for (int k = 0; k < 3; ++k) scale[k] = sah_scale(cmin[k], cmax[k]);
    int bcnt[3][SAH_BINS];
    int32_t blo[3][SAH_BINS][3], bhi[3][SAH_BINS][3];
    for (int k = 0; k < 3; ++k)
        for (int j = 0; j < SAH_BINS; ++j) {
            bcnt[k][j] = 0;
            for (int c = 0; c < 3; ++c) {
                blo[k][j][c] = f2o(inf);
                bhi[k][j][c] = f2o(-inf);
            }
        }
    for (int i = 0; i < cnt; ++i) {
        const float *bx = pb + 6 * (size_t)perm[items[i]];
        for (int k = 0; k < 3; ++k) {
            const int j = sah_bin(centroid2(bx, k), cmin[k], scale[k]);
            ++bcnt[k][j];
            for (int c3 = 0; c3 < 3; ++c3) {
                const int32_t ol = f2o(bx[c3]), oh = f2o(bx[3 + c3]);
                if (ol < blo[k][j][c3]) blo[k][j][c3] = ol;
                if (oh > bhi[k][j][c3]) bhi[k][j][c3] = oh;
            }
        }
    }
    /* sah_choose: the plane after bin `lane` splits the bins 0 .. lane from lane + 1 .. 31 */
    float cost = inf;
    int best = 0;
    for (int lane = 0; lane < SAH_BINS - 1; ++lane)
        for (int k = 0; k < 3; ++k) {
            int pc = 0, rc = 0;
            float plo[3] = {inf, inf, inf}, phi[3] = {-inf, -inf, -inf}, rlo[3] = {inf, inf, inf}, rhi[3] = {-inf, -inf, -inf};
            for (int j = 0; j < SAH_BINS; ++j) {
                const int left = j <= lane;
                if (left) pc += bcnt[k][j];
                else rc += bcnt[k][j];
                for (int c = 0; c < 3; ++c) {
                    if (left) {
                        plo[c] = fminf(plo[c], o2f(blo[k][j][c]));
                        phi[c] = fmaxf(phi[c], o2f(bhi[k][j][c]));
                    }
                    else {
                        rlo[c] = fminf(rlo[c], o2f(blo[k][j][c]));
                        rhi[c] = fmaxf(rhi[c], o2f(bhi[k][j][c]));
                    }
                }
            }
            if (pc > 0 && rc > 0) {
                const float ck = sah_cost(area3(phi[0] - plo[0], phi[1] - plo[1], phi[2] - plo[2]), pc,
                                          area3(rhi[0] - rlo[0], rhi[1] - rlo[1], rhi[2] - rlo[2]), rc);
                const int id = k * 32 + lane;
                if (ck < cost || (ck == cost && id < best)) {
                    cost = ck;
                    best = id;
                }
            }
        }
    /* the node box: the union of all bins (axis 0) */
    for (int c = 0; c < 3; ++c) {
        float lo = inf, hi = -inf;
        for (int j = 0; j < SAH_BINS; ++j) {
            lo = fminf(lo, o2f(blo[0][j][c]));
            hi = fmaxf(hi, o2f(bhi[0][j][c]));
        }
        nb[c] = lo;
        nb[3 + c] = hi;
    }
    int how = 0;
    if (!(cost < inf)) how = 1;
    else if (level + ceil_log2(cnt) >= budget) how = 2;
    if (block) {
        ++C->block_splits;
        if (how == 1) ++C->block_median_coincident;
        if (how == 2) ++C->block_median_budget;
    }
    else {
        ++C->warp_splits;
        if (how == 1) ++C->warp_median_coincident;
        if (how == 2) ++C->warp_median_budget;
    }
    log_task(B, block ? 0 : 1, items, cnt, how ? -1 : best, how, level, budget);
    const int ax = best >> 5, sp = best & 31;
    int *tmp = (int *)malloc(sizeof(int) * (size_t)cnt);
    int l = 0, r = 0;
    for (int i = 0; i < cnt; ++i) {
        int go_left;
        if (how) go_left = i < cnt / 2;
        else {
            const float *bx = pb + 6 * (size_t)perm[items[i]];
            go_left = sah_bin(centroid2(bx, ax), cmin[ax], scale[ax]) <= sp;
        }
        if (go_left) tmp[l++] = items[i];
        else tmp[cnt - 1 - r++] = items[i]; /* the right side fills from the end: reversed */
    }
    memcpy(items, tmp, sizeof(int) * (size_t)cnt);
    free(tmp);
    return l;
}

static void rebuild_subtree(builder *B, int root, int a, int m, int depth_root)
{
    const int ni = B->ni;
    const int budget = 63 - depth_root;
    int alloc = a + 1;
    int *buf = (int *)malloc(sizeof(int) * (size_t)m);
    for (int l = 0; l < m; ++l) buf[l] = a + l;
    task *cur = (task *)malloc(sizeof(task) * (size_t)m), *nxt = (task *)malloc(sizeof(task) * (size_t)m);
    int n_cur = 1, level = 0;
    cur[0].node = root;
    cur[0].cnt = m;
    cur[0].items = buf;
    while (n_cur > 0) {
        int n_nxt = 0;
        for (int t = 0; t < n_cur; ++t) {
            const int node = cur[t].node, cnt = cur[t].cnt;
            int *items = cur[t].items;
            const int nl = split_task(B, node, items, cnt, level, budget);
            const int cb[2] = {0, nl}, ce[2] = {nl, cnt};
            int child[2];
            for (int sd = 0; sd < 2; ++sd) {
                if (ce[sd] - cb[sd] == 1) {
                    const int k = items[cb[sd]];
                    child[sd] = ~k;
                    B->parent2[ni + k] = node;
                }
                else {
                    const int v = alloc++;
                    child[sd] = v;
                    B->parent2[v] = node;
                    nxt[n_nxt].node = v;
                    nxt[n_nxt].cnt = ce[sd] - cb[sd];
                    nxt[n_nxt].items = items + cb[sd];
                    ++n_nxt;
                }
            }
            B->left2[node] = child[0];
            B->right2[node] = child[1];
        }
        task *t = cur;
        cur = nxt;
        nxt = t;
        n_cur = n_nxt;
        ++level;
    }
    free(buf);
    free(cur);
    free(nxt);
}

/* the climbing refit of k_refit_upper (nb = 1, node_box2) and k_refit<2> (nb = 2, node_box01): the second arrival at a
 * node computes its box from its two children */
static void climb(builder *B, int node, int *visit, int nb, float *node_box, const float *leaf_box)
{
    while (node >= 0) {
        if (visit[node]++ == 0) return;
        const int L = B->left2[node], R = B->right2[node];
        for (int e = 0; e < nb; ++e) {
            const float *l6 = L >= 0 ? node_box + 6 * nb * (size_t)L + 6 * e : leaf_box + 6 * nb * (size_t)B->b->perm[~L] + 6 * e;
            const float *r6 = R >= 0 ? node_box + 6 * nb * (size_t)R + 6 * e : leaf_box + 6 * nb * (size_t)B->b->perm[~R] + 6 * e;
            float *o = node_box + 6 * nb * (size_t)node + 6 * e;
            for (int c = 0; c < 3; ++c) {
                o[c] = fminf(l6[c], r6[c]);
                o[3 + c] = fmaxf(l6[3 + c], r6[3 + c]);
            }
        }
        node = B->parent2[node];
    }
}

/* k_collapse4 for the wide node rooted at binary node bnode; returns its canonical index (pre-order) */
static int collapse(builder *B, int bnode, int depth)
{
    orc_wide *w = B->w;
    const int wpn = w->words_per_node;
    const int i = w->n_nodes++;
    if (depth > w->cnt.max_wide_depth) w->cnt.max_wide_depth = depth;
    int ch[4], nc;
    if (B->n == 1) {
        ch[0] = ~0;
        nc = 1;
    }
    else {
        ch[0] = B->left2[bnode];
        ch[1] = B->right2[bnode];
        nc = 2;
        for (int rep = 0; rep < 2; ++rep) {
            int bi = -1;
            float ba = -1.0f;
            for (int c = 0; c < nc; ++c)
                if (ch[c] >= 0) {
                    const float ar = box_area6(B->node_box2 + 6 * (size_t)ch[c]);
                    if (ar > ba) {
                        ba = ar;
                        bi = c;
                    }
                }
            if (bi < 0) break;
            const int bb = ch[bi];
            ch[bi] = B->left2[bb];
            ch[nc++] = B->right2[bb];
        }
    }
    const float pad = B->b->pad;
    float cc[2][3][4], hh[2][3][4];
    int32_t ref[4];
    for (int c = 0; c < 4; ++c) {
        if (c >= nc) {
            for (int e = 0; e < 2; ++e)
                for (int k = 0; k < 3; ++k) {
                    cc[e][k][c] = 0.f;
                    hh[e][k][c] = -INFINITY;
                }
            ref[c] = TRAV_DONE;
            continue;
        }
        const float *bx;
        if (ch[c] >= 0) {
            ref[c] = 0; /* set below, once the child has its index */
            bx = B->motion ? B->node_box01 + 12 * (size_t)ch[c] : B->node_box2 + 6 * (size_t)ch[c];
        }
        else {
            const int slot = ~ch[c];
            const int id = (int)B->b->perm[slot];
            ref[c] = ~((slot << 2) | prim_type(B->s, id));
            bx = B->motion ? B->pbox01 + 12 * (size_t)id : B->b->prim_box + 6 * (size_t)id;
        }
        for (int k = 0; k < 3; ++k) center_half(bx[k], bx[3 + k], pad, &cc[0][k][c], &hh[0][k][c]);
        if (B->motion)
            for (int k = 0; k < 3; ++k) center_half(bx[6 + k], bx[9 + k], pad, &cc[1][k][c], &hh[1][k][c]);
    }
    for (int c = 0; c < nc; ++c)
        if (ch[c] >= 0) ref[c] = collapse(B, ch[c], depth + 1);
    uint32_t *o = w->words + (size_t)wpn * i;
    const int ends = B->motion ? 2 : 1;
    for (int e = 0; e < ends; ++e)
        for (int k = 0; k < 3; ++k) memcpy(o + 12 * e + 4 * k, cc[e][k], 16);
    uint32_t *hw = o + 12 * ends;
    for (int e = 0; e < ends; ++e)
        for (int k = 0; k < 3; ++k)
            for (int p = 0; p < 2; ++p)
                hw[6 * e + 2 * k + p] = (uint32_t)orc_f16_up(hh[e][k][2 * p]) | ((uint32_t)orc_f16_up(hh[e][k][2 * p + 1]) << 16);
    memcpy(o + 18 * ends, ref, 16);
    if (!B->motion) o[22] = o[23] = 0u;
    return i;
}

orc_wide *orc_wide_build(const orc_scene *s, int motion)
{
    const int n = orc_n_objects(s);
    if (n < 1) return NULL;
    orc_bvh *b = orc_bvh_build(s);
    const int ni = n - 1;
    orc_wide *w = (orc_wide *)calloc(1, sizeof(orc_wide));
    builder B;
    memset(&B, 0, sizeof(B));
    B.s = s;
    B.b = b;
    B.n = n;
    B.ni = ni;
    B.motion = motion != 0;
    B.w = w;
    B.nt_shape = n >= 3 ? (n <= 8 * SAH_MAX ? 1024 : 256) : 0;
    w->cnt.sort_small = n <= SMALL_SORT;
    w->cnt.rebuild_shape = B.nt_shape;
    w->words_per_node = B.motion ? 40 : 24;
    const size_t nn = ni > 0 ? (size_t)ni : 1;
    B.left2 = (int32_t *)malloc(4 * nn);
    B.right2 = (int32_t *)malloc(4 * nn);
    B.parent2 = (int32_t *)malloc(4 * (size_t)(2 * n));
    B.node_box2 = (float *)malloc(sizeof(float) * 6 * nn);
    B.node_box01 = (float *)malloc(sizeof(float) * 12 * nn);
    B.pbox01 = (float *)malloc(sizeof(float) * 12 * (size_t)n);
    w->prim_box01 = B.pbox01;
    w->left2 = B.left2;
    w->right2 = B.right2;
    w->node_box2 = B.node_box2;
    /* the traversal-box padding (k_bounds): 2^-20 of the largest coordinate a primitive box or a camera ray can have */
    float mag = 0.0f;
    for (size_t k = 0; k < 6 * (size_t)n; ++k) mag = fmaxf(mag, fabsf(b->prim_box[k]));
    for (int k = 0; k < 3; ++k) mag = fmaxf(mag, fabsf(s->cam.origin[k]) + s->cam.lens_radius);
    w->cnt.pad = mag * 9.5367431640625e-07f;
    for (int id = 0; id < n; ++id) prim_box01(s, id, b->prim_box + 6 * (size_t)id, B.pbox01 + 12 * (size_t)id);
    if (ni > 0) {
        memcpy(B.left2, b->left, 4 * (size_t)ni);
        memcpy(B.right2, b->right, 4 * (size_t)ni);
    }
    memcpy(B.parent2, b->parent, 4 * (size_t)(2 * n - 1));
    for (size_t k = 0; k < 6 * nn; ++k) B.node_box2[k] = NAN; /* every node must be written */
    for (size_t k = 0; k < 12 * nn; ++k) B.node_box01[k] = NAN;

    if (n >= 3) {
        /* ranges (first, last sorted position) and depths of the canonical nodes: children after parents in pre-order */
        int *rlo = (int *)malloc(sizeof(int) * nn), *rhi = (int *)malloc(sizeof(int) * nn), *dep = (int *)malloc(sizeof(int) * nn);
        int *order = (int *)malloc(sizeof(int) * nn), *stk = (int *)malloc(sizeof(int) * nn);
        int no = 0, sp = 0;
        stk[sp++] = 0;
        dep[0] = 0;
        while (sp) {
            const int v = stk[--sp];
            order[no++] = v;
            const int ch[2] = {b->left[v], b->right[v]};
            for (int c = 0; c < 2; ++c)
                if (ch[c] >= 0) {
                    dep[ch[c]] = dep[v] + 1;
                    stk[sp++] = ch[c];
                }
        }
        for (int t = no - 1; t >= 0; --t) {
            const int v = order[t], L = b->left[v], R = b->right[v];
            rlo[v] = L >= 0 ? rlo[L] : ~L;
            rhi[v] = R >= 0 ? rhi[R] : ~R;
        }
        /* k_sah_select: maximal subtrees of 3 .. SAH_MAX leaves */
        int *is_root = (int *)calloc(nn, sizeof(int));
        for (int i = 0; i < ni; ++i) {
            const int size = rhi[i] - rlo[i] + 1, p = b->parent[i];
            const int psize = p >= 0 ? rhi[p] - rlo[p] + 1 : 0x7fffffff;
            if (size >= 3 && size <= SAH_MAX && psize > SAH_MAX) {
                is_root[i] = 1;
                ++w->cnt.n_roots;
                rebuild_subtree(&B, i, rlo[i], size, dep[i]);
            }
        }
        /* k_refit_upper: the uncovered leaves and the subtree roots climb the Morton top */
        int *visit = (int *)calloc(nn, sizeof(int));
        for (int k = 0; k < n; ++k) {
            int p = b->parent[ni + k];
            int size = rhi[p] - rlo[p] + 1, gp = 0;
            if (size == 2 && b->parent[p] >= 0) {
                p = b->parent[p];
                size = rhi[p] - rlo[p] + 1;
                gp = 1;
            }
            if (size >= 3 && size <= SAH_MAX) continue;
            if (gp) ++w->cnt.refit_grandparent;
            else ++w->cnt.refit_parent;
            climb(&B, B.parent2[ni + k], visit, 1, B.node_box2, b->prim_box);
        }
        for (int i = 0; i < ni; ++i)
            if (is_root[i]) climb(&B, B.parent2[i], visit, 1, B.node_box2, b->prim_box);
        free(visit);
        free(is_root);
        free(rlo);
        free(rhi);
        free(dep);
        free(order);
        free(stk);
    }
    else if (ni > 0)
        memcpy(B.node_box2, b->node_box, sizeof(float) * 6 * (size_t)ni);
    if (B.motion && ni > 0) { /* k_refit<2> over the traversal topology */
        int *visit = (int *)calloc(nn, sizeof(int));
        for (int k = 0; k < n; ++k) climb(&B, B.parent2[ni + k], visit, 2, B.node_box01, B.pbox01);
        free(visit);
    }
    /* deepest leaf of the binary traversal tree */
    for (int k = 0; k < n; ++k) {
        int d = 0;
        for (int p = B.parent2[ni + k]; p >= 0; p = B.parent2[p]) ++d;
        if (d > w->cnt.max_binary_depth) w->cnt.max_binary_depth = d;
    }
    w->words = (uint32_t *)calloc((size_t)w->words_per_node * nn, 4);
    collapse(&B, 0, 0);
    free(B.parent2);
    free(B.node_box01);
    orc_bvh_free(b);
    return w;
}

void orc_wide_free(orc_wide *w)
{
    if (!w) return;
    free(w->words);
    free(w->tasks);
    free(w->items);
    free(w->prim_box01);
    free(w->left2);
    free(w->right2);
    free(w->node_box2);
    free(w);
}
