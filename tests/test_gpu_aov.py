"""GPU: the first-hit AOVs (include/rrtb.h rrtb_render_aov) equal the CPU oracle bit for bit in all four buffers -- both
integrators, tree and flat scan, static and moving scenes, edge tiles -- add up over tile shards, tie to the beauty
render, and reach the drop-in's `-A` PFMs unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle_lib import Oracle
from rrt_b200.types import DIFFUSE_LIGHT
from test_aov import AOV_KEYS, aov_bytes, oracle_aov, plane_scene, read_pfm
from test_lights import _scene
from test_moving_instances import fast_spheres_scene, kobj_text, load, scene_text

pytestmark = pytest.mark.gpu

CORNELL = os.path.join(ROOT, "scenes", "cornell.txt")
SEED = 1984


@pytest.fixture(scope="module")
def scenes(tmp_path_factory):
    from rrt_b200 import Scene

    d = tmp_path_factory.mktemp("aov")
    out = {name: load_golden(name)[0] for name in ("final", "test2", "test3")}
    out["cornell"] = Scene.from_file(CORNELL, 97, 61).arrays
    out["fast"] = fast_spheres_scene()  # 64 moving spheres under an open shutter: motion nodes
    out["mobj"] = load(d, scene_text("moving"), name="mobj.txt").arrays
    out["kobj"] = load(d, kobj_text(), name="kobj.txt").arrays
    assert len(out["mobj"].mtriangles) == 8 and len(out["kobj"].mtriangles) > 0
    return out


_oracle_cache = {}


def cached_oracle_aov(scenes, name, W, H, spp, precision):
    """The CPU checker through the oracle's tree (its tree and flat scan give the same bits: tests/test_aov.py)"""
    key = (name, W, H, spp, precision)
    if key not in _oracle_cache:
        _oracle_cache[key] = oracle_aov(Oracle(scenes[name]), W, H, spp, SEED, precision=precision)
    return _oracle_cache[key]


def _diff(got, want):
    for k in AOV_KEYS:
        bad = np.argwhere(got[k].view(np.uint32) != want[k].view(np.uint32))
        if len(bad):
            j, i = bad[0][:2]
            return "%s: %d words differ, first at (j=%d, i=%d): gpu %r oracle %r" % (k, len(bad), j, i, got[k][j, i], want[k][j, i])
    return ""


CASES = [
    ("final", 97, 61, 1), ("final", 97, 61, 7), ("final", 97, 61, 64), ("final", 400, 266, 7),
    ("test2", 97, 61, 64), ("test2", 400, 266, 1),
    ("test3", 97, 61, 7), ("test3", 400, 266, 7),
    ("cornell", 97, 61, 7),
    ("fast", 97, 61, 7), ("fast", 97, 61, 64),
    ("mobj", 97, 61, 7), ("kobj", 97, 61, 64),
]


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("use_bvh", [True, False], ids=["bvh", "scan"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-%dx%d-s%d" % c)
def test_aov_equals_oracle(ctx, scenes, case, use_bvh, precision):
    name, W, H, spp = case
    ctx.set_scene(scenes[name], use_bvh=use_bvh)
    got, st = ctx.render_aov(W, H, spp, SEED, precision=precision)
    want = cached_oracle_aov(scenes, name, W, H, spp, precision)
    assert aov_bytes(got) == aov_bytes(want), _diff(got, want)
    assert st["paths"] == W * H * spp and st["kernel_launches"] == 1


def test_motion_nodes_are_used(ctx, scenes):
    """The `fast` cases above run through motion nodes (40-word nodes), the others through plain ones."""
    ctx.set_scene(scenes["fast"])
    assert ctx.wide_raw().shape[1] == 40
    ctx.set_scene(scenes["final"])
    assert ctx.wide_raw().shape[1] == 24


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_tile_shards_add_up_and_repeat(ctx, scenes, precision):
    W, H, spp = 97, 61, 7
    ctx.set_scene(scenes["test3"])
    whole, _ = ctx.render_aov(W, H, spp, SEED, precision=precision)
    again, _ = ctx.render_aov(W, H, spp, SEED, precision=precision)
    assert aov_bytes(again) == aov_bytes(whole)
    for world in (2, 3):
        total = {k: np.zeros_like(whole[k]) for k in AOV_KEYS}
        paths = 0
        for rank in range(world):
            part, st = ctx.render_aov(W, H, spp, SEED, rank=rank, world=world, precision=precision)
            for k in AOV_KEYS:
                assert not np.any(total[k][part[k] != 0]), (world, rank, k)  # disjoint
                total[k] += part[k]
            paths += st["paths"]
        assert aov_bytes(total) == aov_bytes(whole), world
        assert paths == W * H * spp


def test_rejected_calls_leave_the_context_renderable(ctx, scenes):
    from rrt_b200 import Context, RrtbError

    W, H, spp = 33, 17, 3
    ctx.set_scene(scenes["final"])
    before, _ = ctx.render_aov(W, H, spp, SEED)
    bufs = [np.zeros(3 * W * H, np.float32), np.zeros(3 * W * H, np.float32), np.zeros(W * H, np.float32), np.zeros(W * H, np.float32)]
    ptrs = [C.c_void_p(b.ctypes.data) for b in bufs]
    p = Context.params(W, H, spp, 1, SEED, 0, 2, 1)  # RRTB_SHARD_SAMPLES
    assert ctx.lib.rrtb_render_aov(ctx.h, C.byref(p), *ptrs, None) == -1
    p = Context.params(W, H, spp, 1, SEED)
    for k in range(4):
        q = list(ptrs)
        q[k] = None
        assert ctx.lib.rrtb_render_aov(ctx.h, C.byref(p), *q, None) == -1
    with pytest.raises(RrtbError):
        ctx.render_aov(1, 1, spp, SEED)  # check_render: at least 2x2
    after, _ = ctx.render_aov(W, H, spp, SEED)
    assert aov_bytes(after) == aov_bytes(before)
    img, _ = ctx.render(W, H, spp, 50, SEED)
    assert np.isfinite(img).all() and img.max() > 0


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ["final", "fast", "kobj"])
def test_counters_tie_to_the_beauty_render(ctx, scenes, name, precision):
    """rays = W H spp; hits = the hits of a beauty render at max_depth 1 = sum of coverage x spp"""
    W, H, spp = 97, 61, 7
    ctx.set_scene(scenes[name])
    aov, st = ctx.render_aov(W, H, spp, SEED, count_rays=True, precision=precision)
    _, bst = ctx.render(W, H, spp, 1, SEED, count_rays=True, precision=precision,
                        dtype=np.float64 if precision == "f64" else np.float32)
    assert st["rays"] == W * H * spp == bst["rays"]
    assert st["hits"] == bst["hits"] == int(np.rint(aov["coverage"].astype(np.float64) * spp).sum())
    assert st["box_tests"] > 0 and st["sphere_tests"] + st["msphere_tests"] + st["triangle_tests"] > 0
    plain, _ = ctx.render_aov(W, H, spp, SEED, precision=precision)
    assert aov_bytes(plain) == aov_bytes(aov)  # the counting build computes the same buffers


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_albedo_of_emitters_is_the_beauty_mean(ctx, precision):
    """Emitters with Le <= 1 under a black background: a path ends at its first segment with Le or 0, so the beauty mean
    sum / spp is the mean albedo, to float rounding."""
    W, H, spp = 64, 48, 16
    sc = _scene(W, H, [(DIFFUSE_LIGHT, (0.3, 0.6, 0.9)), (DIFFUSE_LIGHT, (1.0, 0.5, 0.25))],
                [((-0.6, 0, -3), 0.8, 0), ((0.7, 0.2, -4), 1.1, 1)], background=(0.0, 0.0, 0.0))
    ctx.set_scene(sc)
    aov, _ = ctx.render_aov(W, H, spp, SEED, precision=precision)
    img, _ = ctx.render(W, H, spp, 50, SEED, precision=precision, dtype=np.float64)
    mean = img / spp
    cov = aov["coverage"]
    assert 0 < cov.mean() < 1
    assert np.allclose(aov["albedo"], mean, rtol=1e-6, atol=1e-12)


def test_plane_anchor_on_the_gpu(ctx):
    W, H = 16, 12
    sc = plane_scene(W, H)
    ctx.set_scene(sc)
    for precision in ("f32", "f64"):
        got, _ = ctx.render_aov(W, H, 4, 11, precision=precision)
        assert aov_bytes(got) == aov_bytes(oracle_aov(Oracle(sc), W, H, 4, 11, precision=precision))
        assert np.all(got["coverage"] == 1) and np.all(got["albedo"] == np.array([0.2, 0.4, 0.6], np.float32))


@pytest.mark.parametrize("exe, precision, dtype", [("rrt", "f32", np.float32), ("rrtd", "f64", np.float64)])
def test_cli_writes_the_pfms(ctx, tmp_path, exe, precision, dtype):
    from rrt_b200 import Scene

    path = os.path.join(ROOT, "tests", "golden", "scenes", "final.txt")
    W, H, spp = 64, 48, 4
    prefix = str(tmp_path / "p")
    r = subprocess.run([os.path.join(ROOT, "rrt_b200", "bin", exe), "-i", path, "-w", str(W), "-h", str(H), "-s", str(spp),
                        "-o", str(tmp_path / "o.png"), "-A", prefix], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert os.path.exists(tmp_path / "o.png")
    files = {k: read_pfm(prefix + ".%s.pfm" % k) for k in ("color", "albedo", "normal", "depth", "coverage")}
    for k, (lines, _, _) in files.items():
        assert lines == ["PF" if k in ("color", "albedo", "normal") else "Pf", "%d %d" % (W, H), "-1.0"], k
    ctx.set_scene(Scene.from_file(path, W, H))
    sums, _ = ctx.render(W, H, spp, 50, SEED, precision=precision, dtype=dtype)
    want = (sums / np.float32(spp)) if dtype == np.float32 else (sums / float(spp)).astype(np.float32)
    assert files["color"][1].tobytes() == want.astype(np.float32).tobytes()
    aov, _ = ctx.render_aov(W, H, spp, SEED, precision=precision)
    for k in AOV_KEYS:
        assert files[k][1].tobytes() == aov[k].tobytes(), k
