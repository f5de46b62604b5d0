"""The render pinned bit for bit across its launch space (-m gpu).

Every kernel `launch_render` can start is run on a covering list of cases and compared with a plain reference: the
double integrator with the double oracle (oracle/rrt_oracle_f64.c) bit for bit, the float integrator with itself
across schedulers bit for bit and with the float oracle to the usual tolerance.  The cases straddle what the kernels
cut the work into -- 8x4-pixel tiles (edge tiles in x, in y, in both; a single tile; fewer pixels than a warp),
CHUNK = 16 samples of the lane kernel (partial last chunks), a pool's worth of 64-96 slots per warp x 8 warps (far
below and far above) -- and use seeds above 2^32, so that both words of the Philox key matter.

Which case reaches which entry of the two launcher tables of `launch_render` (rrtb_render.cu).  Every case renders
with counting on AND off, so each row below is reached by both instantiations (COUNT_RAYS true / false):

    table   entry                                     reached by (scene of the case; `scan` = set_scene(use_bvh=False))
    lane    [f32][flat scan]                          group 2, every case, `scan`
    lane    [f32][LBVH]                               group 2, every case, RRTB_SCHED_SIMPLE
    lane    [f64][flat scan]                          group 1, every case, `scan`
    lane    [f64][LBVH]                               group 1, every case, RRTB_SCHED_SIMPLE
    pool    [f32, no MTRI][plain nodes]               group 2, final / test2 / test3 (3 moving spheres: no motion nodes),
                                                      varied (final.txt with negative and large fuzz, other indices)
    pool    [f32, no MTRI][motion nodes]              group 2, fast (64 moving spheres, open shutter)
    pool    [f32, MTRI][plain nodes]                  group 2, mtri_closed (8 moving triangles, shutter closed)
    pool    [f32, MTRI][motion nodes]                 group 2, mtri (8 moving triangles, open shutter)
    pool    [f64][plain nodes]                        group 1, final / test2 / test3 / mtri_closed / varied
    pool    [f64][motion nodes]                       group 1, fast / mtri

Groups: (1) double integrator == oracle, (2) float integrator: every scheduler the same bits, (3) tile and sample
shards, (4) knife-edge rays through the 4-wide traversal, (5) the range of the 2^40 fixed-point pixel sums.

The pool's GEN batch decodes (tile, sample) of its items from the first one and wraps at most once to the next group
(rrtb_render_pool.cuh).  With the default thresholds no render reaches that wrap: a warp is only short of work when
all its slots wait in the scatter and gen stacks, so one of them holds >= 32 (a pool has >= 64 slots), every batch
takes 32 items until the queue drains, and the queue head stays a multiple of 32.  Batches of fewer items (and the
wrap) happen in the tuning build with RRTB_TH_SHADE < 32, where groups 1 and 2 also pass.
"""
import numpy as np
import pytest

from conftest import load_golden
from oracle_lib import Oracle
from rrt_b200.types import SceneArrays
from test_gpu_edge_cases import check_wide_tree, make_scene
from test_moving_instances import fast_spheres_scene, load, scene_text
from test_path_by_path import varied_scene
from test_random_scenes import random_scene, special_rays

pytestmark = pytest.mark.gpu

POOL, SIMPLE = 2, 1  # RRTB_SCHED_POOL, RRTB_SCHED_SIMPLE
TILES, SAMPLES = 0, 1  # RRTB_SHARD_*
S0, S1, S2, S3 = 0, 1984, 2**32 + 1984, 2**64 - 1
MAX_SPP = 2**23


def fixed_clamp(spp):
    """The per-sample radiance clamp of a render of spp samples (rrtb_device.cuh fixed_clamp), in plain integers."""
    lg = (spp - 1).bit_length()  # ceil(log2 spp)
    return float(2 ** min(20, 23 - lg))


# ---------------------------------------------------------------------------------------------------------------
# scenes: one per launcher of the pool table, built once
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scenes(tmp_path_factory):
    d = tmp_path_factory.mktemp("launch_space")
    out = {name: load_golden(name)[0] for name in ("final", "test2", "test3")}
    out["fast"] = fast_spheres_scene()
    out["varied"] = varied_scene()
    out["mtri"] = load(d, scene_text("moving"), name="mtri.txt").arrays
    out["mtri_closed"] = load(d, scene_text("moving", 0.5, 0.5), name="mtri_closed.txt").arrays
    assert len(out["mtri"].mtriangles) == 8 and len(out["mtri_closed"].mtriangles) == 8
    return out


# (scene, W, H, spp, max_depth, seed).  Together: every shape of SHAPES, spp of SPPS, depth and seed at least once,
# on every scene; 2x2x1 = 4 paths is far below one pool's worth of slots (>= 64 x 8), 97x61x100 far above it.
CASES = [
    ("final", 97, 61, 100, 50, S1),
    ("final", 33, 17, 17, 50, S0),
    ("final", 9, 5, 33, 2, S2),
    ("final", 2, 2, 1, 50, S3),
    ("final", 31, 3, 16, 1, S1),
    ("final", 8, 4, 15, 50, S2),
    ("final", 97, 61, 1, 2, S0),
    ("test2", 33, 17, 100, 50, S3),
    ("test2", 8, 4, 1, 1, S0),
    ("test2", 9, 5, 16, 50, S1),
    ("test2", 31, 3, 17, 2, S2),
    ("test2", 2, 2, 33, 50, S0),
    ("test2", 97, 61, 15, 50, S2),
    ("test3", 97, 61, 33, 50, S3),
    ("test3", 2, 2, 100, 2, S1),
    ("test3", 31, 3, 1, 50, S2),
    ("test3", 9, 5, 17, 1, S0),
    ("test3", 33, 17, 15, 2, S3),
    ("fast", 97, 61, 17, 50, S2),
    ("fast", 8, 4, 100, 50, S3),
    ("fast", 33, 17, 1, 2, S1),
    ("fast", 31, 3, 33, 50, S0),
    ("fast", 9, 5, 15, 1, S2),
    ("fast", 2, 2, 16, 50, S1),
    ("mtri", 97, 61, 16, 50, S0),
    ("mtri", 33, 17, 33, 50, S2),
    ("mtri", 2, 2, 17, 1, S3),
    ("mtri", 9, 5, 100, 2, S1),
    ("mtri", 31, 3, 15, 50, S1),
    ("mtri_closed", 97, 61, 15, 50, S3),
    ("mtri_closed", 8, 4, 33, 2, S0),
    ("mtri_closed", 33, 17, 100, 50, S2),
    ("mtri_closed", 31, 3, 16, 1, S1),
    ("varied", 97, 61, 17, 50, S2),
    ("varied", 33, 17, 100, 50, S3),
]
SHAPES = {(2, 2), (8, 4), (9, 5), (31, 3), (33, 17), (97, 61)}
SPPS = {1, 15, 16, 17, 33, 100}


def _id(c):
    return "%s-%dx%d-s%d-d%d-seed%d" % c


def test_cases_cover_the_launch_space():
    assert {(c[1], c[2]) for c in CASES} == SHAPES
    assert {c[3] for c in CASES} == SPPS
    assert {c[4] for c in CASES} == {1, 2, 50}
    assert {c[5] for c in CASES} == {S0, S1, S2, S3}
    assert {c[0] for c in CASES} == {"final", "test2", "test3", "fast", "mtri", "mtri_closed", "varied"}
    paths = [c[1] * c[2] * c[3] for c in CASES]
    assert min(paths) < 64 * 8 // 16 and max(paths) > 64 * 8 * 256


def _renders(ctx, scene, W, H, spp, depth, seed, precision, dtype):
    """(label, image, stats) of the pool, the lane kernel over the LBVH and the lane kernel's flat scan, counting on and
    off: every launcher of `launch_render` a scene of this kind reaches in this precision."""
    out = []
    for use_bvh, sched in ((True, POOL), (True, SIMPLE), (False, POOL)):
        ctx.set_scene(scene, use_bvh=use_bvh)
        for count in (True, False):
            img, st = ctx.render(W, H, spp, depth, seed=seed, count_rays=count, scheduler=sched, dtype=dtype, precision=precision)
            out.append(("%s/%s" % ("pool" if use_bvh and sched == POOL else ("lane" if use_bvh else "scan"), "count" if count else "plain"),
                        img, st, count))
    return out


def _where(a, b):
    bad = np.nonzero((a != b).any(axis=-1))
    return "%d pixels differ, first (row, col) %s" % (len(bad[0]), list(zip(bad[0][:4].tolist(), bad[1][:4].tolist())))


# ---------------------------------------------------------------------------------------------------------------
# 1. double integrator: GPU == oracle bit for bit
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=_id)
def test_f64_render_equals_oracle_across_the_launch_space(ctx, scenes, case):
    name, W, H, spp, depth, seed = case
    scene = scenes[name]
    want, _, cnt = Oracle(scene).render_f64(W, H, spp, depth, seed)
    assert cnt["paths"] == W * H * spp
    for label, img, st, count in _renders(ctx, scene, W, H, spp, depth, seed, "f64", np.float64):
        assert img.tobytes() == want.tobytes(), (case, label, _where(img, want))
        assert st["paths"] == cnt["paths"], (case, label)
        if count:
            assert (st["rays"], st["hits"]) == (cnt["rays"], cnt["hits"]), (case, label, st, cnt)


# ---------------------------------------------------------------------------------------------------------------
# 2. float integrator: every scheduler gives the same bits
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=_id)
def test_f32_render_same_bits_on_every_scheduler(ctx, scenes, case):
    name, W, H, spp, depth, seed = case
    scene = scenes[name]
    runs = _renders(ctx, scene, W, H, spp, depth, seed, "f32", np.float32)
    first = runs[0][1]
    counted = [st for _, _, st, count in runs if count]
    for label, img, st, count in runs:
        assert img.tobytes() == first.tobytes(), (case, label, _where(img, first))
        assert st["paths"] == W * H * spp, (case, label)
    assert len({(st["rays"], st["hits"]) for st in counted}) == 1, (case, counted)
    assert counted[0]["rays"] >= W * H * spp
    # against the float oracle: the usual bar.  A single path that a rounding difference sends elsewhere moves a pixel
    # by more than the tolerance, so the bar is a statistic and needs a few hundred pixels to mean anything.
    if W * H >= 500:
        ref, _, cnt = Oracle(scene).render(W, H, spp, depth, seed)
        assert cnt["paths"] == W * H * spp
        a = np.sqrt(first.astype(np.float64) / spp).clip(0, 1)
        b = np.sqrt(ref.astype(np.float64) / spp).clip(0, 1)
        close = np.abs(a - b).max(axis=2) < 1e-3
        assert close.mean() > 0.97, (case, close.mean())
        assert abs(a.mean() - b.mean()) < 2e-3, (case, a.mean(), b.mean())


# ---------------------------------------------------------------------------------------------------------------
# 3. shards
# ---------------------------------------------------------------------------------------------------------------
def shard_paths(W, H, spp, rank, world, mode):
    """Camera paths of one shard, from the tile rule alone: 8x4-pixel tiles t with t % world == rank (all samples), or
    every pixel and the samples s with s % world == rank.  Also the mask of the pixels the shard owns."""
    tiles_x = (W + 7) // 8
    j, i = np.mgrid[0:H, 0:W]
    if mode == TILES:
        own = ((j // 4) * tiles_x + (i // 8)) % world == rank
        return int(own.sum()) * spp, own
    return W * H * len(range(rank, spp, world)), np.ones((H, W), bool)


# (scene, W, H, spp, world, scheduler): 9x5 and 31x3 have 4 tiles, fewer than 7 ranks; spp 3 < 7 ranks
SHARD_CASES = [
    ("final", 33, 17, 5, 3, POOL),
    ("fast", 97, 61, 4, 7, SIMPLE),
    ("test2", 9, 5, 6, 7, POOL),
    ("mtri", 31, 3, 3, 7, POOL),
    ("test3", 33, 17, 17, 2, SIMPLE),
    ("mtri_closed", 97, 61, 2, 3, POOL),
]


@pytest.mark.parametrize("case", SHARD_CASES, ids=lambda c: "%s-%dx%d-s%d-w%d-sched%d" % c)
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_shards_sum_to_the_whole_image(ctx, scenes, case, precision):
    name, W, H, spp, world, sched = case
    scene = scenes[name]
    ctx.set_scene(scene, use_bvh=True)
    seed = S2
    whole, _ = ctx.render(W, H, spp, 50, seed=seed, scheduler=sched, dtype=np.float64, precision=precision)
    if precision == "f64":
        want, _, _ = Oracle(scene).render_f64(W, H, spp, 50, seed)
        assert whole.tobytes() == want.tobytes(), case
    for mode in (TILES, SAMPLES):
        acc = np.zeros_like(whole)
        idle = 0
        for rank in range(world):
            # the double framebuffer: partial sums of fixed-point values add exactly in double at this spp
            part, st = ctx.render(W, H, spp, 50, seed=seed, rank=rank, world=world, shard_mode=mode, count_rays=True,
                                  scheduler=sched, dtype=np.float64, precision=precision)
            paths, own = shard_paths(W, H, spp, rank, world, mode)
            assert st["paths"] == paths, (case, mode, rank, st["paths"], paths)
            assert not part[~own].any(), (case, mode, rank)  # pixels of other ranks' tiles are exactly 0
            if paths == 0:
                idle += 1
                assert not part.any() and st["rays"] == 0, (case, mode, rank)
            if mode == TILES:  # the float framebuffer of a tile shard is the whole image's on the owned pixels
                part32, _ = ctx.render(W, H, spp, 50, seed=seed, rank=rank, world=world, shard_mode=mode, scheduler=sched,
                                       precision=precision)
                assert part32[own].tobytes() == whole[own].astype(np.float32).tobytes() and not part32[~own].any()
            acc += part
        assert acc.tobytes() == whole.tobytes(), (case, mode, _where(acc, whole))
        n_tiles = ((W + 7) // 8) * ((H + 3) // 4)
        assert idle == (max(world - n_tiles, 0) if mode == TILES else max(world - spp, 0)), (case, mode, idle)


def test_shard_cases_include_idle_ranks():
    assert any(w > ((W + 7) // 8) * ((H + 3) // 4) for _, W, H, _, w, _ in SHARD_CASES)
    assert any(w > spp for _, _, _, spp, w, _ in SHARD_CASES)
    assert {w for *_, w, _ in SHARD_CASES} == {2, 3, 7}


# ---------------------------------------------------------------------------------------------------------------
# 4. knife-edge rays through the GPU's 4-wide traversal
# ---------------------------------------------------------------------------------------------------------------
def pad_magnitude(ctx, scene):
    """M of the traversal-box padding 2^-20 M (rrtb_bvh.cu k_bounds): the largest coordinate of a canonical primitive
    box, or |camera origin| + lens radius on an axis."""
    box = ctx.bvh_arrays()["prim_box"].astype(np.float64)
    cam = scene.camera
    lens = float(cam["lens_radius"][0])
    return max(float(np.abs(box).max()), float((np.abs(cam["origin"][0].astype(np.float64)) + lens).max()))


def face_rays(ctx, scene, n, seed):
    """Rays whose origin lies exactly on a face of a canonical primitive box and that run along that face (the direction
    component across the face is 0; a third of them run along an edge of the face)."""
    rng = np.random.default_rng(seed)
    box = ctx.bvh_arrays()["prim_box"]
    k = rng.integers(0, len(box), size=n)
    lo, hi = box[k, :3].astype(np.float64), box[k, 3:].astype(np.float64)
    o = lo + rng.uniform(0, 1, size=(n, 3)) * (hi - lo)
    axis = rng.integers(0, 3, size=n)
    side = rng.integers(0, 2, size=n).astype(bool)
    rows = np.arange(n)
    o[rows, axis] = np.where(side, hi[rows, axis], lo[rows, axis])  # exactly the face's coordinate
    d = rng.normal(size=(n, 3))
    d[rows, axis] = 0.0
    edge = rng.uniform(size=n) < 1 / 3
    d[rows[edge], (axis[edge] + 1) % 3] = 0.0
    r = np.zeros((n, 7), np.float32)
    r[:, 0:3] = np.clip(o.astype(np.float32), box[k, :3], box[k, 3:])  # on the face after the rounding to float too
    r[rows, axis] = np.where(side, box[k, 3 + axis], box[k, axis])
    r[:, 3:6] = d
    r[:, 6] = rng.uniform(scene.camera["time0"][0], max(scene.camera["time1"][0], 1e-3), size=n)
    return r


def secondary_rays(ids, rec, rays, seed):
    """Rays leaving hit points the GPU returned: a lambertian-like bounce, the mirror direction and a direction in the
    tangent plane of the hit (grazing its own surface)."""
    rng = np.random.default_rng(seed)
    m = ids >= 0
    p, nrm, d = rec[m, 0:3].astype(np.float64), rec[m, 3:6].astype(np.float64), rays[m, 3:6].astype(np.float64)
    n = len(p)
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    lam = nrm + 0.999 * u
    mir = d - 2 * np.sum(d * nrm, axis=1, keepdims=True) * nrm
    tan = u - np.sum(u * nrm, axis=1, keepdims=True) * nrm
    out = []
    for dirs in (lam, mir, tan):
        r = np.zeros((n, 7), rays.dtype)
        r[:, 0:3] = p
        r[:, 3:6] = dirs
        r[:, 6] = rays[m, 6]
        out.append(r)
    r = np.concatenate(out)
    return r[np.abs(r[:, 3:6]).max(axis=1) > 0]


def axis_quads(seed, n=10):
    """n axis-aligned squares (two triangles each) with integer corners and sides of 2 or 4: their boxes are exact in
    float and their half extents (1 or 2, and 0 across the square) exact in fp16, so the traversal boxes of these leaves
    are as tight as the padding alone makes them -- no rounding of the box to fp16 hides a padding that is too small."""
    from rrt_b200.types import triangle_dtype

    rng = np.random.default_rng(seed + 9000)
    t = np.zeros(2 * n, triangle_dtype)
    for q in range(n):
        a = q % 3
        u, v = (a + 1) % 3, (a + 2) % 3
        side = float(rng.choice([2, 4]))
        p0 = np.zeros(3)
        p0[a] = rng.integers(-6, 7)
        p0[u], p0[v] = rng.integers(-6, 6 - int(side) + 1, size=2)
        du, dv = np.zeros(3), np.zeros(3)
        du[u], dv[v] = side, side
        m = int(rng.integers(0, 5))
        t[2 * q] = (p0, p0 + du, p0 + du + dv, m)
        t[2 * q + 1] = (p0, p0 + du + dv, p0 + dv, m)
    return t


def quad_rays(tris, n, seed):
    """Rays from random origins to random points of the axis-aligned squares (interiors, edges and corners)."""
    rng = np.random.default_rng(seed + 9100)
    k = rng.integers(0, len(tris), size=n)
    v0, v1, v2 = (tris[f][k].astype(np.float64) for f in ("v0", "v1", "v2"))
    w = rng.dirichlet((1, 1, 1), size=n)
    w[: n // 4, 0] = 0.0  # on the diagonal edge v1 v2 (the two triangles' shared edge)
    w[: n // 4] /= w[: n // 4].sum(axis=1, keepdims=True)
    w[n // 4: n // 2] = np.eye(3)[rng.integers(0, 3, size=n // 2 - n // 4)]  # corners
    p = w[:, 0:1] * v0 + w[:, 1:2] * v1 + w[:, 2:3] * v2
    r = np.zeros((n, 7), np.float32)
    r[:, 0:3] = rng.uniform(-9, 9, size=(n, 3))
    r[:, 3:6] = p - r[:, 0:3]
    return r


def _tight(scene, seed):
    """The random scene without its radius-500 ground sphere (padding 2^-20 M with M ~ 12 instead of ~ 1000), with
    axis-aligned squares whose leaf boxes only the padding makes thicker than zero."""
    tri = np.concatenate([scene.triangles, axis_quads(seed)])
    return SceneArrays(scene.camera, scene.materials, scene.spheres[1:].copy(), scene.mspheres, tri, scene.mtriangles)


def _proxy(scene, seed):
    """A stand-in for special_rays, which aims at static spheres other than the first and at static triangles: the
    moving spheres / triangles of `scene` at the middle of the shutter (the rays are traced at that time)."""
    from rrt_b200.types import sphere_dtype, triangle_dtype

    mid = 0.5 * (scene.camera["time0"][0] + scene.camera["time1"][0])
    sp = [scene.spheres[:1]] if len(scene.spheres) else [np.zeros(1, sphere_dtype)]
    ms = scene.mspheres
    if len(ms):
        s = np.zeros(len(ms), sphere_dtype)
        f = ((mid - ms["time0"]) / (ms["time1"] - ms["time0"]))[:, None]
        s["center"] = ms["center0"] + f * (ms["center1"] - ms["center0"])
        s["radius"] = ms["radius"]
        sp.append(s)
    sp.append(scene.spheres[1:])
    tris = [scene.triangles]
    mt = scene.mtriangles
    if len(mt):
        t = np.zeros(len(mt), triangle_dtype)
        f = ((mid - mt["time0"]) / (mt["time1"] - mt["time0"]))[:, None]
        t["v0"] = mt["v0"] + f * mt["delta"]
        t["v1"] = mt["v1"] + f * (mt["delta"] + mt["extra1"])
        t["v2"] = mt["v2"] + f * (mt["delta"] + mt["extra2"])
        tris.append(t)
    tri = np.concatenate(tris)
    if len(tri) == 0:
        tri = random_scene(seed).triangles
    return SceneArrays(scene.camera, scene.materials, np.concatenate(sp), None, tri)


def _same(label, a, b):
    for k, (x, y) in enumerate(zip(a, b)):
        if x.tobytes() != y.tobytes():
            bad = np.nonzero((x != y).reshape(len(x), -1).any(axis=1))[0]
            pytest.fail("%s: output %d differs on %d rays, first %s" % (label, k, len(bad), bad[:8].tolist()))


def _knife_edge_scene(scenes, which, seed):
    if which == "random":
        return random_scene(40 + seed)
    if which == "tight":
        return _tight(random_scene(40 + seed), seed)
    return scenes[which]


@pytest.mark.parametrize("seed", range(2))
@pytest.mark.parametrize("which", ["random", "tight", "fast", "mtri"])
def test_knife_edge_rays_through_the_traversal(ctx, scenes, which, seed):
    """Closest hits of the 4-wide traversal == the GPU's flat scan == the oracle's flat scan, bit for bit (ids, t and the
    7-float record), float and double.  Contract: ray origins lie within the padding magnitude M, the largest scene
    coordinate or |camera| + lens radius on an axis -- true of every ray a render makes (camera rays start in the lens,
    bounces at hit points).  Rays here that start farther out are dropped.  Scenes: (a) random, (b) tight: (a) without
    its ground sphere and with axis-aligned squares, (c) 64 fast spheres (motion nodes), (d) 8 moving triangles."""
    scene = _knife_edge_scene(scenes, which, seed)
    ctx.set_scene(scene, use_bvh=True)
    check_wide_tree(ctx, scene.n_objects)
    orc = Oracle(scene)
    M = pad_magnitude(ctx, scene)
    if which == "tight":
        assert M < 20.0  # 2^-20 M ~ 1e-5: a slab test that is not conservative shows here
    base = random_scene(40 + seed)
    if which == "random":
        rays = special_rays(seed, base)
    elif which == "tight":  # the same rays (special_rays skips the first sphere, the ground), plus the squares
        rays = special_rays(seed, SceneArrays(base.camera, base.materials, base.spheres, base.mspheres, scene.triangles))
        rays = np.concatenate([rays, quad_rays(scene.triangles[len(base.triangles):], 4000, seed)])
    else:  # aimed at this scene's moving primitives where they are at mid-shutter, and traced then
        rays = special_rays(seed, _proxy(scene, seed))
        mid = 0.5 * (scene.camera["time0"][0] + scene.camera["time1"][0])
        timed = rays.copy()
        rays[:, 6] = mid
        rays = np.concatenate([rays, timed])
    rays = np.concatenate([rays, face_rays(ctx, scene, 6000, seed)])
    rays = rays[np.abs(rays[:, 0:3]).max(axis=1) <= M]
    assert len(rays) > 5000
    a = ctx.trace(rays, 0.001, "bvh", want_rec=True)
    _same("%s f32 bvh vs scan" % which, a, ctx.trace(rays, 0.001, "scan", want_rec=True))
    _same("%s f32 bvh vs oracle scan" % which, a, orc.trace(rays, 0.001, "scan", want_rec=True))
    assert (a[0] >= 0).mean() > 0.1 and (a[0] < 0).any()
    r64 = rays.astype(np.float64)
    a64 = ctx.trace_f64(r64, 0.001, "bvh", want_rec=True)
    _same("%s f64 bvh vs scan" % which, a64, ctx.trace_f64(r64, 0.001, "scan", want_rec=True))
    _same("%s f64 bvh vs oracle scan" % which, a64, orc.trace_f64(r64, 0.001, "scan", want_rec=True))
    # secondary-style rays from the GPU's own hit points, in each precision
    sec = secondary_rays(a[0], a[2], rays, seed)
    sec = sec[np.abs(sec[:, 0:3]).max(axis=1) <= M]
    b = ctx.trace(sec, 0.001, "bvh", want_rec=True)
    _same("%s f32 secondary bvh vs scan" % which, b, ctx.trace(sec, 0.001, "scan", want_rec=True))
    _same("%s f32 secondary bvh vs oracle scan" % which, b, orc.trace(sec, 0.001, "scan", want_rec=True))
    sec64 = secondary_rays(a64[0], a64[2], r64, seed)
    sec64 = sec64[np.abs(sec64[:, 0:3]).max(axis=1) <= M]
    b64 = ctx.trace_f64(sec64, 0.001, "bvh", want_rec=True)
    _same("%s f64 secondary bvh vs scan" % which, b64, ctx.trace_f64(sec64, 0.001, "scan", want_rec=True))
    _same("%s f64 secondary bvh vs oracle scan" % which, b64, orc.trace_f64(sec64, 0.001, "scan", want_rec=True))
    assert (b[0] >= 0).any() and (b64[0] >= 0).any()


# ---------------------------------------------------------------------------------------------------------------
# 5. the range of the 2^40 fixed-point pixel sums
# ---------------------------------------------------------------------------------------------------------------
def test_fixed_clamp_rule():
    assert [fixed_clamp(s) for s in (1, 2, 8, 9, 16, 17, 64, 4096, 2**22 + 1, 2**23)] == \
        [2.0**20, 2.0**20, 2.0**20, 2.0**19, 2.0**19, 2.0**18, 2.0**17, 2.0**11, 1.0, 1.0]
    for spp in list(range(1, 3000)) + [2**k + d for k in range(12, 24) for d in (-1, 0, 1) if 2**k + d <= MAX_SPP]:
        assert spp * fixed_clamp(spp) * 2.0**40 <= 2.0**63  # no pixel sum can wrap, whatever the albedos


def test_spp_beyond_the_fixed_point_range_is_rejected(ctx):
    import torch

    from rrt_b200 import RrtbError

    ctx.set_scene(make_scene(spheres=[((0, 0.5, 0), 1.0, 0)]))
    W, H = 8, 4
    acc = torch.zeros(3 * W * H, dtype=torch.int64, device="cuda")
    ctx.frame_create(W, H)
    for spp in (MAX_SPP + 1, 2**24, 2**24 + 2**20, 2**31 - 1):
        calls = [lambda: ctx.render(W, H, spp, 1),
                 lambda: ctx.render(W, H, spp, 1, dtype=np.float64, precision="f64"),
                 lambda: ctx.render_device(ctx.params(W, H, spp, 1), acc.data_ptr()),
                 lambda: ctx.render_shard(ctx.params(W, H, spp, 1, 1984, 0, 2, SAMPLES))]
        for k, call in enumerate(calls):
            with pytest.raises(RrtbError) as e:
                call()
            assert e.value.status == -1, (spp, k)  # RRTB_ERR_INVALID
    torch.cuda.synchronize()
    assert not acc.any()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_sky_sums_at_the_largest_spp(ctx, precision):
    """A 2x2 image that sees only sky (its one sphere is behind the camera), one segment per path, 2^23 samples: the
    largest spp accepted.  Sky radiance is below 1 per channel (blue: 1), so the sums are spp times the sky colour."""
    ctx.set_scene(make_scene(spheres=[((0, 0.5, 40), 1.0, 0)]), use_bvh=True)
    W, H, spp = 2, 2, MAX_SPP
    imgs = []
    for sched in (POOL, SIMPLE):
        img, st = ctx.render(W, H, spp, 1, seed=S2, count_rays=True, scheduler=sched, dtype=np.float64, precision=precision)
        assert st["paths"] == W * H * spp and st["rays"] == W * H * spp and st["hits"] == 0
        s = img / spp
        assert np.all((s[..., 0] >= 0.5) & (s[..., 0] <= 1.0)), s
        assert np.all((s[..., 1] >= 0.7) & (s[..., 1] <= 1.0)), s
        assert np.all(np.abs(s[..., 2] - 1.0) <= 1e-6), s
        imgs.append(img)
    assert imgs[0].tobytes() == imgs[1].tobytes()
    # the same render as a sample shard over 3 ranks of one context, added in the frame's 64-bit sum buffer
    ctx.frame_create(W, H, f64=True)
    for rank in range(3):
        st = ctx.render_shard(ctx.params(W, H, spp, 1, S2, rank, 3, SAMPLES, precision=precision))
        assert st["paths"] == W * H * len(range(rank, spp, 3))
    got = ctx.frame_download(np.empty((H, W, 3), np.float64), SAMPLES)
    assert got.tobytes() == imgs[0].tobytes()


def gain_scene():
    """final.txt with every lambertian and metal albedo multiplied by 3: a path's throughput grows at every bounce,
    and single samples reach the per-sample clamp."""
    sc, _ = load_golden("final")
    m = sc.materials.copy()
    g = (m["type"] == 0) | (m["type"] == 1)
    m["albedo"][g] *= 3
    return SceneArrays(sc.camera, m, sc.spheres, sc.mspheres, sc.triangles, sc.mtriangles)


@pytest.mark.parametrize("W,H,spp", [(97, 61, 64), (16, 8, 4096)])
def test_gain_scene_equals_oracle_and_stays_in_range(ctx, W, H, spp):
    scene = gain_scene()
    want, fixed, _ = Oracle(scene).render_f64(W, H, spp, 50, S1)
    C = fixed_clamp(spp)
    assert int(fixed.max()) <= spp * int(C) * 2**40  # the oracle's sums obey the bound too
    for use_bvh, sched in ((True, POOL), (True, SIMPLE), (False, POOL)):
        ctx.set_scene(scene, use_bvh=use_bvh)
        img, _ = ctx.render(W, H, spp, 50, seed=S1, scheduler=sched, dtype=np.float64, precision="f64")
        assert img.tobytes() == want.tobytes(), (spp, use_bvh, sched, _where(img, want))
        assert img.max() <= spp * C
        f32, _ = ctx.render(W, H, spp, 50, seed=S1, scheduler=sched, dtype=np.float64)
        assert f32.max() <= spp * C


@pytest.mark.parametrize("spp", [64, 4096, MAX_SPP])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_gain_scene_samples_reach_the_clamp(ctx, spp, precision):
    """Rank 0 of a sample shard of `spp` ranks renders sample 0 of every pixel, clamped for a render of `spp` samples;
    a 1-spp render is the same sample under the clamp 2^20.  The first must be the second clamped to fixed_clamp(spp)
    exactly -- and some pixels must really be clamped."""
    scene = gain_scene()
    ctx.set_scene(scene, use_bvh=True)
    W, H = 97, 61
    C = fixed_clamp(spp)
    for sched in (POOL, SIMPLE):
        one, _ = ctx.render(W, H, 1, 50, seed=S1, scheduler=sched, dtype=np.float64, precision=precision)
        part, st = ctx.render(W, H, spp, 50, seed=S1, rank=0, world=spp, shard_mode=SAMPLES, scheduler=sched,
                              dtype=np.float64, precision=precision)
        assert st["paths"] == W * H
        assert (one > C).sum() >= 3, (spp, float(one.max()))
        assert part.tobytes() == np.minimum(one, C).tobytes(), (spp, sched, _where(part, np.minimum(one, C)))
