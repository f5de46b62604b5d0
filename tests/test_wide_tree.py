"""The 4-wide traversal tree pinned bit for bit against a CPU reference (oracle/rrt_oracle_wide.c).

Every render kernel walks the tree that rrtb_bvh.cu builds from the canonical LBVH: k_sah_select / k_sah_rebuild
rebuild its lower subtrees with a binned SAH, k_refit_upper refits the Morton top, k_collapse4 collapses the result to
4-wide nodes (float centres, fp16 half extents rounded up).  Closest hits do not depend on that tree, so a wrong split,
tie rule, rounding or padding changes no image -- only speed.  Here the tree itself is compared with a reference that
restates the build in float in the GPU's operation order, on scenes that straddle every size threshold of the build.

CPU part: the reference reaches every row of the threshold table below, its trees are partitions whose stored boxes are
exactly the encoded unions of their primitives' boxes, its split choices are the cheapest wherever float64 costs tell
the candidates apart, its outputs are pinned by SHA-256, and the PTX of the build kernels does not depend on -fmad.
GPU part (-m gpu): the GPU's raw nodes, renumbered canonically (pre-order, children in slot order), equal the
reference's word for word; rebuilds give the same tree; closest hits through the tree equal the flat scans.

    threshold                                               reached by / avoided by (counters of the reference)
    SMALL_SORT = 2048: bitonic sort or radix sort           sort_small: n2048 / n2049
    SAH_MAX = 512: whole-scene subtree or Morton top        n_roots == 1 and no climbing leaves: n512 / n513
    8 * SAH_MAX = 4096: k_sah_rebuild<1024> or <256>        rebuild_shape: n4096 / n4097
    SAH_BIG = 128: block-wide split (1024 shape only)       block_splits: n129 / n128; warp splits of runs > 128: n4097
    cnt <= 4: exact enumeration                             small_splits: spheres3 / spheres2
    median split: coincident centroids or depth budget      *_median_coincident: coincident (block and warp);
                                                            *_median_budget: deep_budget (block and warp)
    parent / grandparent rule of k_refit_upper              refit_parent: outlier; refit_grandparent: outlier_pair
    n == 1, n < 3 (no rebuild)                              spheres1, spheres2 / spheres3
    motion nodes (>= 8 moving, open shutter)                msph8, mtri8 / msph7, mtri8_closed
    fp16 +inf and subnormal half extents                    ground1e5, tiny
"""
import hashlib
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle_lib import Oracle, camera_derive, f16_up
from rrt_b200.types import SceneArrays, material_dtype, msphere_dtype, mtriangle_dtype, sphere_dtype, triangle_dtype

TRAV_DONE = np.uint32(0x80000000)
SAH_MAX = 512


# ---------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------
def _mats():
    m = np.zeros(3, material_dtype)
    m["type"] = [0, 1, 2]
    m["albedo"][0] = (0.6, 0.5, 0.4)
    m["albedo"][1] = (0.8, 0.8, 0.9)
    m["param"] = [0, 0.2, 1.5]
    return m


def _cam(lookfrom=(0, 3, 14), lookat=(0, 0.5, 0), shutter=(0.0, 0.0)):
    return camera_derive(lookfrom, lookat, (0, 1, 0), 40.0, 1.5, 0.05, 10.0, *shutter)


def _spheres(centers, radii, seed=0):
    s = np.zeros(len(centers), sphere_dtype)
    s["center"] = np.asarray(centers, np.float32)
    s["radius"] = np.asarray(radii, np.float32)
    s["material"] = np.random.default_rng(seed).integers(0, 3, size=len(centers))
    return s


def random_spheres(n, seed, extent=6.0):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-extent, extent, size=(n, 3)).astype(np.float32)
    r = np.exp(rng.uniform(np.log(0.02), np.log(0.4), size=n)).astype(np.float32)
    return SceneArrays(_cam(), _mats(), _spheres(c, r, seed))


def row_of_spheres(n):
    return SceneArrays(_cam(), _mats(), _spheres([(2.0 * k, 0.5, 0.0) for k in range(n)], [0.5] * n))


def cluster_and_far(n_far, seed=11):
    """600 spheres in a cluster and n_far (1 or 2) spheres far from it: the far ones hang off the root of more than 512
    leaves directly (one sphere) or as a 2-leaf node (two)."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-2, 2, size=(600, 3))
    far = [(40.0, 40.0, 40.0), (40.5, 40.0, 40.0)][:n_far]
    c = np.concatenate([c, far]).astype(np.float32)
    r = np.full(len(c), 0.05, np.float32)
    return SceneArrays(_cam(), _mats(), _spheres(c, r, seed))


def coincident(n=600):
    """n spheres with one centre: every binned split falls back to the median, and every Morton code is the same."""
    return SceneArrays(_cam(), _mats(), _spheres(np.tile([(0.0, 0.5, 0.0)], (n, 1)), 0.1 + 0.001 * np.arange(n)))


def degenerate_triangles(n=300, seed=5):
    """Triangles whose three vertices coincide, at points of one line parallel to the x axis: every box, and every union
    of boxes, has extent along x only and surface area 0, so every SAH cost is 0 and only the tie rules decide the
    tree."""
    rng = np.random.default_rng(seed)
    t = np.zeros(n, triangle_dtype)
    p = np.zeros((n, 3), np.float32)
    p[:, 0] = rng.uniform(-5, 5, size=n)
    p[:, 1:] = (0.5, -1.0)
    t["v0"], t["v1"], t["v2"] = p, p, p
    return SceneArrays(_cam(), _mats(), np.zeros(0, sphere_dtype), None, t)


def ground_1e5(seed=3):
    """A radius-1e5 ground sphere: its half extents (and the root's) pass 65504 and are stored as fp16 +inf."""
    sc = random_spheres(40, seed)
    s = sc.spheres.copy()
    s[0] = ((0.0, -100000.5, 0.0), 100000.0, 0)
    return SceneArrays(sc.camera, sc.materials, s)


def tiny_triangles(n=40, seed=4):
    """Triangles of extent ~1e-7 near the origin seen from a camera at distance ~1: the padding is 2^-20 of ~1, so the
    leaves' half extents are fp16 subnormals, rounded up."""
    rng = np.random.default_rng(seed)
    t = np.zeros(n, triangle_dtype)
    base = rng.uniform(-0.3, 0.3, size=(n, 3))
    t["v0"] = base
    t["v1"] = base + rng.uniform(-1e-7, 1e-7, size=(n, 3))
    t["v2"] = base + rng.uniform(-1e-7, 1e-7, size=(n, 3))
    cam = camera_derive((0, 0, 0.9), (0, 0, 0), (0, 1, 0), 60.0, 1.5, 0.0, 1.0)
    return SceneArrays(cam, _mats(), np.zeros(0, sphere_dtype), None, t)


def deep_comb(n=2048):
    """Centroids on the Morton grid (spheres of radius 0.25 at q + 0.5 in grid units, grid = 1023.5 / 1024): one sphere
    in the code-0 cell at each power-of-two object id (1, 2, .., 1024) and at id 0, one at code 2^j for j = 0..29, and
    the remaining ids in the far corner (codes with bit 29 set).  Sorted by (code, id), the keys make the Karras tree a
    comb: the path to id 0 splits at code bits 29 .. 0 and then at id bits 10 .. 0."""
    pow2 = [0] + [1 << i for i in range(11) if (1 << i) < n]
    comb = comb_codes()
    rng = np.random.default_rng(2)
    c = np.zeros((n, 3))
    fill = [k for k in range(n) if k not in pow2]
    c[pow2] = 0.0
    c[pow2[1:]] = rng.uniform(0.0, 0.4, size=(len(pow2) - 1, 3))  # id 0 at the origin: the centroid minimum
    c[fill[:30]] = comb
    c[fill[30:]] = rng.uniform(768.0, 1023.0, size=(len(fill) - 30, 3))
    c[fill[-1]] = 1023.5  # the centroid maximum on every axis
    cam = camera_derive((512, 512, 3000), (512, 512, 0), (0, 1, 0), 40.0, 1.0, 0.0, 3000.0)
    return SceneArrays(cam, _mats(), _spheres(c.astype(np.float32), np.full(n, 0.25, np.float32)))


def comb_codes():
    """Centres (q + 0.5 in grid units) of the Morton codes 2^j, j = 0..29: code bit j is bit j // 3 of the quantised
    x (j % 3 == 2), y (1) or z (0)"""
    comb = []
    for j in range(30):
        p = [0.5, 0.5, 0.5]
        p[2 - j % 3] = (1 << (j // 3)) + 0.5
        comb.append(p)
    return comb


def deep_budget(m=600, ratio=1.2):
    """The Morton comb (codes 2^j, each a leaf directly under a node of more than 512 leaves) ending in a cluster of m
    spheres in the code-0 cell, at x = 0.9 ratio^-k: the cluster's subtrees are rebuilt from depth ~31 with a budget of
    ~32 levels, and the binned SAH of an exponential row splits off a few spheres at a time, so the depth budget forces
    median splits (the farthest centres underflow to 0 and coincide).  The rebuilt tree reaches binary depth 63."""
    x = 0.9 * ratio ** -np.arange(m, dtype=np.float64)
    cl = np.zeros((m, 3))
    cl[:, 0] = x
    c = np.concatenate([cl, comb_codes(), [[1023.5] * 3]])
    r = np.concatenate([np.maximum(x * 0.01, 1e-30), np.full(31, 0.25)])  # no radius underflows to 0
    cam = camera_derive((512, 512, 3000), (512, 512, 0), (0, 1, 0), 40.0, 1.0, 0.0, 3000.0)
    return SceneArrays(cam, _mats(), _spheres(c.astype(np.float32), r.astype(np.float32)))


def moving_spheres(n, shutter=(0.0, 1.0), seed=7):
    rng = np.random.default_rng(seed)
    ms = np.zeros(n, msphere_dtype)
    c0 = rng.uniform(-3, 3, size=(n, 3)).astype(np.float32)
    ms["center0"], ms["center1"] = c0, c0 + rng.uniform(-1, 1, size=(n, 3)).astype(np.float32)
    ms["time0"], ms["time1"] = 0.0, 1.0
    ms["radius"] = 0.2
    ms["material"] = rng.integers(0, 3, size=n)
    s = _spheres([(0.0, -1000.0, 0.0), (0.5, 1.0, 0.0)], [1000.0, 0.5])
    return SceneArrays(_cam(shutter=shutter), _mats(), s, ms)


def moving_triangles(n=8, shutter=(0.0, 1.0), seed=8):
    rng = np.random.default_rng(seed)
    t = np.zeros(n, mtriangle_dtype)
    v0 = rng.uniform(-2, 2, size=(n, 3))
    t["v0"], t["v1"], t["v2"] = v0, v0 + rng.uniform(-1, 1, size=(n, 3)), v0 + rng.uniform(-1, 1, size=(n, 3))
    t["delta"] = rng.uniform(-0.5, 0.5, size=(n, 3))
    t["extra1"] = rng.uniform(-0.2, 0.2, size=(n, 3))
    t["extra1"][: n // 2] = 0.0  # half of them translate only
    t["time0"], t["time1"] = 0.0, 1.0
    t["material"] = rng.integers(0, 3, size=n)
    s = _spheres([(0.0, -1000.0, 0.0)], [1000.0])
    return SceneArrays(_cam(shutter=shutter), _mats(), s, None, np.zeros(0, triangle_dtype), t)


def cornell():
    from rrt_b200 import Scene

    return Scene.from_file(os.path.join(ROOT, "scenes", "cornell.txt"), 24, 16).arrays


SCENES = {
    **{"spheres%d" % n: (lambda n=n: row_of_spheres(n)) for n in (1, 2, 3, 4, 5)},
    **{"n%d" % n: (lambda n=n: random_spheres(n, n)) for n in (128, 129, 512, 513, 2047, 2048, 2049, 4096, 4097)},
    "outlier": lambda: cluster_and_far(1),
    "outlier_pair": lambda: cluster_and_far(2),
    "coincident": coincident,
    "degenerate": degenerate_triangles,
    "ground1e5": ground_1e5,
    "tiny": tiny_triangles,
    "deep_comb": deep_comb,
    "deep_budget": deep_budget,
    "msph7": lambda: moving_spheres(7),
    "msph8": lambda: moving_spheres(8),
    "mtri8": lambda: moving_triangles(8),
    "mtri8_closed": lambda: moving_triangles(8, shutter=(0.5, 0.5)),
    "final": lambda: load_golden("final")[0],
    "test2": lambda: load_golden("test2")[0],
    "test3": lambda: load_golden("test3")[0],
    "cornell": cornell,
}


def motion_rule(scene):
    """The library's rule for motion nodes (rrtb_api.cu use_motion_nodes): 8 moving primitives or more, open shutter"""
    cam = scene.camera
    return len(scene.mspheres) + len(scene.mtriangles) >= 8 and cam["time0"][0] != cam["time1"][0]


_cache = {}


def reference(name):
    """(scene, reference tree) of one scene of SCENES, built once per session"""
    if name not in _cache:
        scene = SCENES[name]()
        _cache[name] = (scene, Oracle(scene).wide_tree(motion_rule(scene)))
    return _cache[name]


# ---------------------------------------------------------------------------------------------------------------
# reading the words
# ---------------------------------------------------------------------------------------------------------------
def decode(words):
    """(centres [m, ends, 3, 4] float32, half words [m, ends, 3, 4] uint16, refs [m, 4] int32) of raw nodes"""
    m, wpn = words.shape
    ends = 2 if wpn == 40 else 1
    c = words[:, :12 * ends].copy().view(np.float32).reshape(m, ends, 3, 4)
    hw = words[:, 12 * ends:18 * ends].reshape(m, ends, 3, 2)
    h = np.stack([hw & 0xFFFF, hw >> 16], axis=-1).reshape(m, ends, 3, 4).astype(np.uint16)
    ref = words[:, 18 * ends:18 * ends + 4].view(np.int32)
    return c, h, ref


def canonical(words):
    """The nodes renumbered in pre-order from the root (node 0), children in slot order, internal refs rewritten"""
    m, wpn = words.shape
    ends = 2 if wpn == 40 else 1
    ref = words[:, 18 * ends:18 * ends + 4].view(np.int32)
    order, stack = [], [0]
    while stack:
        v = stack.pop()
        order.append(v)
        stack.extend(int(r) for r in ref[v][::-1] if r >= 0)
    assert sorted(order) == list(range(m)), "the nodes do not form one tree"
    new = np.empty(m, np.int64)
    new[order] = np.arange(m)
    out = words[order].copy()
    r = out[:, 18 * ends:18 * ends + 4].view(np.int32)
    r[r >= 0] = new[r[r >= 0]]
    return out


def half_up(h):
    """float32 -> fp16 bits rounded toward +inf, in numpy (independent of orc_f16_up): round to nearest, then step up
    where that landed below"""
    h = np.asarray(h, np.float32)
    with np.errstate(over="ignore"):
        r = h.astype(np.float16)
    low = r.astype(np.float64) < h.astype(np.float64)
    r[low] = np.nextafter(r[low], np.float16(np.inf))
    return r.view(np.uint16)


def encode_box(lo, hi, pad):
    """center_half in float32 numpy: c = 0.5 (lo + hi), h = max(hi - c, c - lo) + pad, h as fp16 rounded up"""
    f = np.float32
    lo, hi = np.asarray(lo, f), np.asarray(hi, f)
    c = (f(0.5) * (lo + hi)).astype(f)
    h = (np.maximum((hi - c).astype(f), (c - lo).astype(f)) + f(pad)).astype(f)
    return c, half_up(h)


def tree_of(words):
    """(parent, slot, depth) of every node of canonically numbered words"""
    _, _, ref = decode(words)
    m = len(ref)
    parent = np.full(m, -1)
    depth = np.zeros(m, np.int64)
    for v in range(m):
        for r in ref[v]:
            if r >= 0:
                assert r > v
                parent[r] = v
                depth[r] = depth[v] + 1
    return parent, depth


# ---------------------------------------------------------------------------------------------------------------
# CPU: the reference
# ---------------------------------------------------------------------------------------------------------------
def test_scene_list_reaches_every_threshold(built_lib):
    """Each path of the build is taken by some scene of SCENES and avoided by another (the table of the docstring)."""
    cnt = {name: reference(name)[1]["counters"] for name in SCENES}
    tasks = {name: reference(name)[1]["tasks"] for name in SCENES}
    n = {name: reference(name)[0].n_objects for name in SCENES}

    def both(pred):
        hit = [k for k in SCENES if pred(k)]
        assert hit and len(hit) < len(SCENES), hit
        return hit

    assert cnt["n2048"]["sort_small"] == 1 and cnt["n2049"]["sort_small"] == 0
    both(lambda k: cnt[k]["sort_small"])
    assert cnt["n4096"]["rebuild_shape"] == 1024 and cnt["n4097"]["rebuild_shape"] == 256
    assert cnt["spheres2"]["rebuild_shape"] == 0 and cnt["spheres3"]["rebuild_shape"] == 1024
    both(lambda k: cnt[k]["rebuild_shape"] == 256)
    # whole-scene subtree or Morton top
    for k in ("n512", "n128", "n129", "final"):
        assert cnt[k]["n_roots"] == 1 and cnt[k]["refit_parent"] + cnt[k]["refit_grandparent"] == 0, k
    assert cnt["n513"]["n_roots"] >= 2
    both(lambda k: n[k] > SAH_MAX)
    # SAH_BIG: the block path, and runs of more than 128 on warps in the 256 shape
    assert cnt["n129"]["block_splits"] >= 1 and cnt["n128"]["block_splits"] == 0 and cnt["n128"]["warp_splits"] >= 1
    assert cnt["n4096"]["block_splits"] >= 1 and cnt["n4097"]["block_splits"] == 0
    assert ((tasks["n4097"][:, 0] == 1) & (tasks["n4097"][:, 2] > 128)).any()
    both(lambda k: cnt[k]["block_splits"])
    # exact small splits: spheres3 .. 5 at the root, none below 3 primitives
    assert cnt["spheres3"]["small_splits"] >= 1 and cnt["spheres2"]["small_splits"] == 0
    assert cnt["spheres5"]["warp_splits"] == 1  # the root run of 5
    both(lambda k: cnt[k]["small_splits"])
    # median fallbacks
    assert cnt["coincident"]["block_median_coincident"] >= 1 and cnt["coincident"]["warp_median_coincident"] >= 1
    both(lambda k: cnt[k]["block_median_coincident"] + cnt[k]["warp_median_coincident"])
    both(lambda k: cnt[k]["block_median_budget"] + cnt[k]["warp_median_budget"])
    assert cnt["deep_budget"]["block_median_budget"] >= 1 and cnt["deep_budget"]["warp_median_budget"] >= 1
    assert cnt["deep_budget"]["max_binary_depth"] == 63
    # k_refit_upper: parent rule and grandparent rule
    assert cnt["outlier"]["refit_parent"] == 1 and cnt["outlier"]["refit_grandparent"] == 0
    assert cnt["outlier_pair"]["refit_grandparent"] == 2 and cnt["outlier_pair"]["refit_parent"] == 0
    both(lambda k: cnt[k]["refit_parent"])
    both(lambda k: cnt[k]["refit_grandparent"])
    # motion nodes
    wpn = {k: reference(k)[1]["words"].shape[1] for k in SCENES}
    assert wpn["msph8"] == wpn["mtri8"] == 40 and wpn["msph7"] == wpn["mtri8_closed"] == 24
    both(lambda k: wpn[k] == 40)
    # fp16 extremes
    half = {k: decode(reference(k)[1]["words"])[1] for k in SCENES}
    assert (half["ground1e5"] == 0x7C00).any() and not (half["n512"] == 0x7C00).any()
    sub = lambda k: ((half[k] & 0x7C00) == 0) & ((half[k] & 0x3FF) != 0)
    assert sub("tiny").any() and not sub("final").any()


@pytest.mark.parametrize("name", list(SCENES))
def test_reference_tree_is_an_exact_encoding_of_the_unions(name, built_lib):
    """The reference's tree is a partition of the primitives (every sorted position once, every node but the root the
    child of one earlier node), every stored child box is exactly the encoding of the exact union of its primitives'
    boxes (not merely enclosing it), unused slots are (0, -inf, TRAV_DONE), and the depth fits the traversal stack."""
    scene, w = reference(name)
    orc = Oracle(scene)
    bvh = orc.bvh_arrays()
    n = scene.n_objects
    words = w["words"]
    cnt = w["counters"]
    # the padding, 2^-20 of the largest coordinate a primitive box or a camera ray can have (k_bounds), in float32
    f = np.float32
    cam = scene.camera[0]
    mag = max(f(np.abs(bvh["prim_box"]).max()), max(f(abs(f(o)) + f(cam["lens_radius"])) for o in cam["origin"]))
    assert cnt["pad"] == bvh["pad"] == f(f(mag) * f(2.0**-20))
    assert np.array_equal(canonical(words), words)  # already in canonical order
    c, h, ref = decode(words)
    m, ends = len(words), c.shape[1]
    assert m <= max(n - 1, 1)
    parent, depth = tree_of(words)
    assert int(depth.max()) == cnt["max_wide_depth"] <= cnt["max_binary_depth"] <= 63
    assert 3 * cnt["max_wide_depth"] + 1 <= 192  # RRTB_STACK: a visit pushes at most 3 entries
    used = ref != np.int32(TRAV_DONE.view(np.int32))
    assert np.all(c[:, :, :, :][np.broadcast_to(~used[:, None, None, :], c.shape)] == 0)
    assert np.all(h[np.broadcast_to(~used[:, None, None, :], h.shape)] == 0xFC00)  # fp16 -inf
    leaf = used & (ref < 0)
    slots = (~ref[leaf]) >> 2
    assert np.array_equal(np.sort(slots), np.arange(n))
    assert np.array_equal(np.sort(ref[used & (ref >= 0)]), np.arange(1, m))
    perm = bvh["perm"]
    ns, nms, nt = len(scene.spheres), len(scene.mspheres), len(scene.triangles)
    types = np.select([perm < ns, perm < ns + nms, perm < ns + nms + nt], [0, 1, 2], 3)
    assert np.array_equal((~ref[leaf]) & 3, types[slots])
    # exact unions, deepest node first
    pb = (w["prim_box01"] if ends == 2 else bvh["prim_box"])[perm].reshape(n, ends, 6)
    lo = np.full((m, 4, ends, 3), np.inf, np.float32)
    hi = np.full((m, 4, ends, 3), -np.inf, np.float32)
    li, lk = np.nonzero(leaf)
    lo[li, lk], hi[li, lk] = pb[(~ref[li, lk]) >> 2, :, :3], pb[(~ref[li, lk]) >> 2, :, 3:]
    for v in np.argsort(-depth, kind="stable"):
        if parent[v] >= 0:
            k = int(np.nonzero(ref[parent[v]] == v)[0][0])
            lo[parent[v], k], hi[parent[v], k] = lo[v].min(axis=0), hi[v].max(axis=0)
    wc, wh = encode_box(lo, hi, cnt["pad"])  # [m, 4, ends, 3]
    wc, wh = np.transpose(wc, (0, 2, 3, 1)), np.transpose(wh, (0, 2, 3, 1))  # [m, ends, 3, 4]
    u = np.broadcast_to(used[:, None, None, :], c.shape)
    assert np.array_equal(c[u].view(np.uint32), wc[u].view(np.uint32))
    assert np.array_equal(h[u], wh[u])


def area64(lo, hi):
    e = hi.astype(np.float64) - lo.astype(np.float64)
    return e[..., 0] * e[..., 1] + e[..., 1] * e[..., 2] + e[..., 2] * e[..., 0]


@pytest.mark.parametrize("name", list(SCENES))
def test_reference_picks_the_cheapest_split(name, built_lib):
    """Every split of the reference, re-evaluated in float64 from the primitive boxes: all 2^(cnt-1) - 1 partitions of a
    run of 2..4 boxes, all 93 planes of a binned run (bins recomputed here from float32 centroids).  Where the float64
    costs separate the candidates by more than the float32 rounding of the costs, the reference took the cheapest; a
    median split happens exactly where no plane has primitives on both sides or the depth budget ran out."""
    scene, w = reference(name)
    bvh = Oracle(scene).bvh_arrays()
    pb = bvh["prim_box"][bvh["perm"]]  # sorted-position order
    f = np.float32
    checked = 0
    # the depth budget of each rebuilt subtree: 63 - canonical depth of its root, the node whose leaves are the run of
    # its first task (level 0)
    lo_leaf, depth = canonical_ranges(bvh)
    budget_of = {}
    for path, first, cnt, choice, how, level, budget in w["tasks"]:
        if level == 0:
            run = w["items"][first:first + cnt]
            node = [v for v in range(len(depth)) if lo_leaf[v] == (run.min(), run.max())]
            assert len(node) == 1 and budget == 63 - depth[node[0]], (run.min(), run.max(), budget)
            budget_of.update({int(k): int(budget) for k in run})
    for path, first, cnt, choice, how, level, budget in w["tasks"]:
        assert budget == budget_of[int(w["items"][first])]
        box = pb[w["items"][first:first + cnt]]
        if path == 2:  # exact: element 0 always on the left
            masks = 1 | (np.arange((1 << (cnt - 1)) - 1) << 1)
            costs = []
            for mk in masks:
                left = ((mk >> np.arange(cnt)) & 1).astype(bool)
                costs.append(area64(box[left, :3].min(0), box[left, 3:].max(0)) * left.sum()
                             + area64(box[~left, :3].min(0), box[~left, 3:].max(0)) * (~left).sum())
            costs = np.array(costs)
            assert how == (2 if level + cnt - 1 >= budget else 0)  # every cost of 2..4 finite boxes is finite
            if how:
                assert choice == (1 << (cnt // 2)) - 1
                continue
            got = costs[list(masks).index(choice)]
            if np.all(costs == costs[0]):  # a tie between all candidates: the lowest mask
                assert choice == masks[0]
        else:
            c2 = (box[:, :3] + box[:, 3:]).astype(f)
            cmin, cmax = c2.min(0), c2.max(0)
            with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
                scale = np.where(cmax > cmin, f(32) / (cmax - cmin).astype(f), f(0)).astype(f)
                x = ((c2 - cmin).astype(f) * scale).astype(f)
            # cvt.rzi.s32.f32: NaN (0 x inf, a scale that overflowed) -> 0, saturating
            b = np.minimum(31, np.trunc(np.nan_to_num(x, nan=0.0, posinf=2.0**31)).astype(np.int64))
            costs = np.full((3, 31), np.inf)
            for k in range(3):
                for s in range(31):
                    left = b[:, k] <= s
                    if left.all() or not left.any():
                        continue
                    costs[k, s] = (area64(box[left, :3].min(0), box[left, 3:].max(0)) * left.sum()
                                   + area64(box[~left, :3].min(0), box[~left, 3:].max(0)) * (~left).sum())
            assert (how == 1) == (not np.isfinite(costs).any())
            if how != 1:
                assert how == (2 if level + int(cnt - 1).bit_length() >= budget else 0)
            if how:
                assert choice == -1
                continue
            got = costs[choice >> 5, choice & 31]
            assert np.isfinite(got)
            fin = costs[np.isfinite(costs)]
            if np.all(fin == fin[0]):  # a tie between all candidates: the lowest axis * 32 + bin
                k, sb = np.nonzero(np.isfinite(costs))
                assert choice == int((k * 32 + sb).min())
        best = costs.min()
        assert got <= best + 1e-6 * got + 1e-30, (path, cnt, got, best)
        checked += 1
    assert checked or scene.n_objects < 3


def canonical_ranges(bvh):
    """((first, last) sorted position, depth) of every internal node of the canonical LBVH"""
    left, right = bvh["left"], bvh["right"]
    ni = len(left)
    rng, depth = [None] * ni, [0] * ni
    order, stack = [], [0] if ni else []
    while stack:
        v = stack.pop()
        order.append(v)
        for c in (left[v], right[v]):
            if c >= 0:
                depth[c] = depth[v] + 1
                stack.append(c)
    for v in reversed(order):
        a = (~left[v], ~left[v]) if left[v] < 0 else rng[left[v]]
        b = (~right[v], ~right[v]) if right[v] < 0 else rng[right[v]]
        rng[v] = (min(a[0], b[0]), max(a[1], b[1]))
    return rng, depth


def area32(b):
    """box_area6 in float32, each product and sum rounded once: x*y + y*z + z*x"""
    f = np.float32
    x, y, z = f(b[3] - b[0]), f(b[4] - b[1]), f(b[5] - b[2])
    return f(f(f(x * y) + f(y * z)) + f(z * x))


@pytest.mark.parametrize("name", list(SCENES))
def test_reference_collapse_opens_the_largest_child(name, built_lib):
    """The reference's binary traversal tree has exact unions as node boxes, and its 4-wide nodes are the greedy collapse
    of it: from the two children of a binary node, twice open the internal child of largest surface area (first maximum
    in slot order wins; the opened node's left child takes its slot, its right child the next free one).  The collapse is
    redone here in numpy, in pre-order, and must give the reference's child refs."""
    scene, w = reference(name)
    bvh = Oracle(scene).bvh_arrays()
    n = scene.n_objects
    left, right, box = w["left2"], w["right2"], w["node_box2"]
    pb = bvh["prim_box"][bvh["perm"]]
    if n >= 2:  # node boxes: exact unions of the primitive boxes below
        def union(v):
            parts = [pb[~c] if c < 0 else union(c) for c in (left[v], right[v])]
            u = np.concatenate([np.minimum(parts[0][:3], parts[1][:3]), np.maximum(parts[0][3:], parts[1][3:])])
            assert np.array_equal(box[v], u), v
            return u
        union(0)
    _, _, ref = decode(w["words"])
    nxt = [0]

    def wide(b):
        i = nxt[0]
        nxt[0] += 1
        ch = [~0] if n == 1 else [int(left[b]), int(right[b])]
        for _ in range(2 if n > 1 else 0):
            bi, ba = -1, np.float32(-1)
            for c, x in enumerate(ch):
                if x >= 0 and area32(box[x]) > ba:
                    bi, ba = c, area32(box[x])
            if bi < 0:
                break
            bb = ch[bi]
            ch[bi] = int(left[bb])
            ch.append(int(right[bb]))
        for c, x in enumerate(ch):
            if x < 0:
                assert ref[i, c] < 0 and (~ref[i, c]) >> 2 == ~x, (i, c)
            else:
                assert ref[i, c] == wide(x), (i, c)
        assert np.all(ref[i, len(ch):] == np.int32(TRAV_DONE.view(np.int32)))
        return i

    wide(0)
    assert nxt[0] == len(ref)


def test_f16_round_up_is_exact():
    """orc_f16_up (the reference's fp16 round-up in integer arithmetic) against numpy: normal, subnormal, overflow and
    signed values, and every float just around each fp16 value."""
    rng = np.random.default_rng(1)
    hs = np.arange(0, 0x7C00, dtype=np.uint16).view(np.float16).astype(np.float32)
    vals = np.concatenate([hs, np.nextafter(hs, np.float32(np.inf)), np.nextafter(hs, np.float32(-np.inf)),
                           rng.uniform(0, 70000, 2000).astype(np.float32), np.float32(2.0) ** rng.uniform(-40, 17, 2000).astype(np.float32),
                           np.array([65504, 65504.004, 65519.996, 65520, 1e6, 1e-45, 3e-8, 5.960464e-08, 6.1035156e-05], np.float32)])
    vals = np.concatenate([vals, -vals[::7]]).astype(np.float32)
    vals = vals[::5] if len(vals) > 30000 else vals
    got = np.array([f16_up(v) for v in vals], np.uint16)
    assert np.array_equal(got, half_up(vals))
    assert f16_up(float("inf")) == 0x7C00 and f16_up(float("-inf")) == 0xFC00



# computed with this file's scenes; a change of the build or of the reference changes them
WIDE_PINS = {
    'spheres1': 'ae7e0458f63636ce89112a83a6e0edb017a0332b79bd9c19a6f62929569f8a88',
    'spheres2': '17e333725804ee0c15f21705c3be0160baf3b5f51b9cdf8af0977362155f9eea',
    'spheres3': '35d59c5c4203e7470ce23459c508fd6255e3116075e8af05c501fb1677a455c1',
    'spheres4': '7bac8acc5d44032d1bd8a32ff767b1a346441e7079e05dfa3e9d510ec07cef22',
    'spheres5': 'b910618c957ea4097e55f4485ddaf791d81f18b06756f6e4a542ca00895ffbdb',
    'n128': '556c0af0466a8351eebd5b7ed0298c2d1a3cf90aa037c343cf5d142c1af49197',
    'n129': 'c506e72ae071865b6d2c84b7a00d19ff725be11d8dcaff6e573659b8ade91b50',
    'n512': '34bc2b3fa248ad2d6d1ab8cd4d6d74bd28057248ea7f171eb3778e74ee32a257',
    'n513': '9ed59ab1a3aa9e9e6ad10c775ef09a6e4d25453f1172b73aa7899eccdf06d2b8',
    'n2047': 'd7d35ece35d31835d05997ac8c31444dca0a11acfaae832bebc01d2fc9c190d3',
    'n2048': 'cf78884f30e90b725a643bfac4c6e91e54af5b74b225ec03df6a297ad94246ad',
    'n2049': '1bcf56a596374f28889838b1cd3e8f9931888ca3bf76327728a80376a60534bb',
    'n4096': 'f9578e510dd08e6408494e6739aacefa1e3b2356c0e00823d4f164d810d4fd8e',
    'n4097': '736604f32065e40edc28f8ffdca83d6ff279cd3f76e37d93e9960c67e354760a',
    'outlier': '22b8e4e15cec3c3b4211f26efb189f20da863415f294e7eff9659c58bd511ffd',
    'outlier_pair': '5bd94edf0e881ef0d89fb447e76c6434bd47a5d7e0f73f6b8a210e338e101a4a',
    'coincident': '017c569e8758dc8c11c7a65655a7388f3d4f86a9850e928dc4f3bd7e2ee8105f',
    'degenerate': 'da9e5e2ca15d9b163ae8025575466bff63e4f215b84164bcd17f6537e6338220',
    'ground1e5': 'e5e92b6f1bc19d877aeec19d5b5dd69b27cd397f27dee68b408c948506df6457',
    'tiny': '10d3a506830ad69a566d6c0a716b8f6945a2bf00a875a398d690110ced07049a',
    'deep_comb': '6009987c0ccdea6e8382c633f48cfe5b762f44e4f70c1158dcf2f74a0eb35ede',
    'deep_budget': '8a6147bbde82104b311f515427272e36353e6b16f3896fc4fc692e2b1bb1c82f',
    'msph7': '4fba03cf05ee44bbceadd8203ebc7abed245536f0abbf738f9dfb4a30c4a64a7',
    'msph8': '5ee9453cfebf826eb7375ad068025aa3dcf57919f9fb762d2731e745792ce493',
    'mtri8': 'ff0f5a1b7c92aabb7d34ec43d0e7a3efe2fb1f8d800e9e37ba9dabfcb04f7f4a',
    'mtri8_closed': '568aa52c55afad9683f1d09dfa2debdd71f2d31578f73975eeb1c8a6a275e40b',
    'final': '28f28d8f58d9d7e34b9e8463be307052f11075b61f522d49dabf0b4c986dacf6',
    'test2': '9faa102780818913a507c9e5cffe199ed9f8d527761b17d7bbafddc09389f3f4',
    'test3': 'f2167c2c3afb0472c700aa9b906067728debfc8d3d03eee282f4b4972d036041',
    'cornell': 'ade8c3b5665a6dab716b0d151d05891fea446f8c03fa55d05ad9481a4883112a',
}


def wide_digest(w):
    cnt = dict(w["counters"])
    return hashlib.sha256(w["words"].tobytes() + json.dumps(cnt, sort_keys=True).encode()).hexdigest()


@pytest.mark.parametrize("name", list(SCENES))
def test_reference_outputs_are_pinned(name, built_lib):
    """SHA-256 of the reference's canonical words and counters per scene"""
    assert wide_digest(reference(name)[1]) == WIDE_PINS[name]


def test_deep_comb_reaches_its_depth(built_lib):
    """The comb's canonical LBVH reaches depth 41 (code bits 29 .. 0, then id bits 10 .. 0): the deepest path a Karras
    tree of 2048 primitives can have, 30 + ceil(log2 n) levels.  Its rebuilt traversal tree stays within the budget."""
    scene, w = reference("deep_comb")
    b = Oracle(scene).bvh_arrays()
    assert set(b["morton"][[1 << i for i in range(11)]]) == {0} and b["morton"][0] == 0
    assert sorted(np.unique(b["morton"])[:31].tolist()) == [0] + [1 << j for j in range(30)]
    parent, n = b["parent"], scene.n_objects
    d = 0
    p = parent[n - 1 + int(np.nonzero(b["perm"] == 0)[0][0])]
    while p >= 0:
        d, p = d + 1, parent[p]
    assert d == 41
    assert w["counters"]["max_binary_depth"] <= 63 and w["counters"]["max_wide_depth"] <= 63


def test_ptx_of_the_build_kernels_does_not_depend_on_fma_contraction(tmp_path):
    """Every product and sum of the tree build rounds once by its source: the PTX of the kernels that compute boxes,
    costs and encodings is the same under nvcc -fmad=true and -fmad=false (so ptxas contracts nothing there)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "rrt_b200", "csrc")
    kernels = {"k_sah_rebuild<1024>": "_ZN4rrtb13k_sah_rebuildILi1024EEEv", "k_sah_rebuild<256>": "_ZN4rrtb13k_sah_rebuildILi256EEEv",
               "k_collapse4": "_ZN4rrtb11k_collapse4E", "k_refit_upper": "_ZN4rrtb13k_refit_upperE",
               "k_refit<1>": "_ZN4rrtb7k_refitILi1EEEv", "k_refit<2>": "_ZN4rrtb7k_refitILi2EEEv", "k_bounds": "_ZN4rrtb8k_boundsE"}
    procs = {}
    for fmad in ("true", "false"):
        out = tmp_path / ("bvh_%s.ptx" % fmad)
        procs[fmad] = (out, subprocess.Popen([nvcc, "-std=c++17", "-O3", "--expt-relaxed-constexpr", "-gencode", "arch=compute_100a,code=sm_100a",
                                              "-fmad=" + fmad, "-ptx", os.path.join(csrc, "rrtb_bvh.cu"), "-o", str(out)]))
    bodies = {}
    for fmad, (out, p) in procs.items():
        assert p.wait(timeout=600) == 0
        lines = out.read_text().splitlines()
        bodies[fmad] = {}
        for name, mangled in kernels.items():
            i = next(k for k, ln in enumerate(lines) if ".entry " + mangled in ln)
            j = next(k for k in range(i, len(lines)) if lines[k] == "}")
            bodies[fmad][name] = lines[i:j + 1]
    for name in kernels:
        assert bodies["true"][name] == bodies["false"][name], name
        assert not any("fma.rn.f32" in ln for ln in bodies["true"][name]), name


# ---------------------------------------------------------------------------------------------------------------
# GPU: the device's tree is the reference's
# ---------------------------------------------------------------------------------------------------------------
def check_gpu_tree(ctx, scene, w):
    got, want = ctx.bvh_arrays(), Oracle(scene).bvh_arrays()
    for k in ("morton", "perm", "left", "right", "parent", "node_box", "prim_box"):
        assert got[k].tobytes() == want[k].tobytes(), k
    raw = ctx.wide_raw()
    assert raw.shape == w["words"].shape, (raw.shape, w["words"].shape)
    can = canonical(raw)
    if not np.array_equal(can, w["words"]):
        bad = np.nonzero((can != w["words"]).any(axis=1))[0]
        pytest.fail("%d of %d nodes differ from the reference, first %s" % (len(bad), len(can), bad[:8].tolist()))
    return can


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_gpu_tree_equals_the_reference(ctx, name):
    """Canonical LBVH == the oracle; the GPU's raw nodes renumbered canonically == the reference, word for word; a second
    upload and a rebuild forced by rrtb_camera_set (a camera farther out: a larger padding) give the reference's tree."""
    scene, w = reference(name)
    ctx.set_scene(scene, use_bvh=True)
    first = check_gpu_tree(ctx, scene, w)
    ctx.set_scene(scene, use_bvh=True)
    assert np.array_equal(canonical(ctx.wide_raw()), first)
    cam = scene.camera.copy()
    cam["origin"] = cam["origin"] * np.float32(2.0) + np.float32(3.0)
    far = SceneArrays(cam, scene.materials, scene.spheres, scene.mspheres, scene.triangles, scene.mtriangles,
                      background=scene.background)
    ctx.set_camera(cam)
    check_gpu_tree(ctx, far, Oracle(far).wide_tree(motion_rule(far)))


def aimed_rays(ctx, scene, n, seed):
    """Rays from random origins to random points of random primitive boxes, at random times of the camera's shutter"""
    rng = np.random.default_rng(seed)
    box = ctx.bvh_arrays()["prim_box"].astype(np.float64)
    k = rng.integers(0, len(box), size=n)
    p = box[k, :3] + rng.uniform(0, 1, size=(n, 3)) * (box[k, 3:] - box[k, :3])
    r = np.zeros((n, 7), np.float32)
    r[:, 0:3] = rng.uniform(-9, 9, size=(n, 3))
    r[:, 3:6] = p - r[:, 0:3]
    r[:, 6] = rng.uniform(scene.camera["time0"][0], scene.camera["time1"][0], size=n)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_gpu_closest_hits_through_the_tree(ctx, name):
    """Closest hits through the tree == the GPU flat scan == the oracle scan, float and double, on knife-edge rays
    (special_rays, rays along faces of primitive boxes) whose origins lie within the padding magnitude M"""
    from test_gpu_launch_space import _same, face_rays, pad_magnitude
    from test_random_scenes import special_rays

    scene, _ = reference(name)
    ctx.set_scene(scene, use_bvh=True)
    orc = Oracle(scene)
    M = pad_magnitude(ctx, scene)
    rays = [face_rays(ctx, scene, 4000, 1), aimed_rays(ctx, scene, 4000, 2)]
    if len(scene.spheres) > 1 and len(scene.triangles):
        rays.append(special_rays(1, scene))
    rays = np.concatenate(rays)
    rays = rays[np.abs(rays[:, 0:3]).max(axis=1) <= M]
    if len(rays) > 20000:
        rays = rays[np.random.default_rng(0).choice(len(rays), 20000, replace=False)]
    a = ctx.trace(rays, 0.001, "bvh", want_rec=True)
    _same("%s f32 bvh vs scan" % name, a, ctx.trace(rays, 0.001, "scan", want_rec=True))
    _same("%s f32 bvh vs oracle scan" % name, a, orc.trace(rays, 0.001, "scan", want_rec=True))
    r64 = rays.astype(np.float64)
    a64 = ctx.trace_f64(r64, 0.001, "bvh", want_rec=True)
    _same("%s f64 bvh vs scan" % name, a64, ctx.trace_f64(r64, 0.001, "scan", want_rec=True))
    _same("%s f64 bvh vs oracle scan" % name, a64, orc.trace_f64(r64, 0.001, "scan", want_rec=True))
    if name not in ("degenerate", "tiny"):  # degenerate triangles are never hit, the tiny ones rarely
        assert (a[0] >= 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["deep_comb", "deep_budget"])
def test_gpu_deep_trees_render_the_same_bits(ctx, name):
    """On the deepest trees: the pool, the lane kernel and the flat scan render the same bits, and the debug build (if
    built) counts no violated traversal-stack bound"""
    import ctypes as C
    import sys

    scene, _ = reference(name)
    ctx.set_scene(scene, use_bvh=True)
    imgs = [ctx.render(40, 24, 4, 8, seed=5, scheduler=s)[0] for s in (2, 1)]
    ctx.set_scene(scene, use_bvh=False)
    imgs.append(ctx.render(40, 24, 4, 8, seed=5)[0])
    assert imgs[0].tobytes() == imgs[1].tobytes() == imgs[2].tobytes()
    assert imgs[0].any()
    dbg = os.path.join(ROOT, "rrt_b200", "librrtb200_dbg.so")
    if not os.path.exists(dbg):
        return
    code = r'''
import sys, ctypes as C
import numpy as np
sys.path[:0] = [%r, %r]
from test_wide_tree import reference
from rrt_b200 import Context
from rrt_b200.types import Stats
ctx = Context(0)
ctx.set_scene(reference(%r)[0], True)
worst = 0
for sched in (1, 2):
    for prec in ("f32", "f64"):
        p = ctx.params(40, 24, 4, 8, 5, scheduler=sched, precision=prec)
        out = np.empty((24, 40, 3), np.float32)
        st = Stats()
        assert ctx.lib.rrtb_render(ctx.h, C.byref(p), C.c_void_p(out.ctypes.data), C.byref(st)) == 0
        worst = max(worst, st.reserved)
print("violations", worst)
''' % (ROOT, os.path.join(ROOT, "tests"), name)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=dict(os.environ, RRTB_LIB=dbg))
    assert r.returncode == 0, r.stderr[-800:]
    assert "violations 0" in r.stdout, r.stdout

