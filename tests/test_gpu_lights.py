"""-m gpu: diffuse_light emitters and a constant background on the B200 (the LIGHTS kernels of launch_render).

  G1  the analytic anchors of tests/test_lights.py give the same exact sums on the GPU, both integrators, on the pool,
      RRTB_SCHED_SIMPLE and the flat scan, counting on and off; the clamp anchor sums to spp * fixed(2)
  G2  final.txt plus an emitter deep inside its ground sphere: the LIGHTS kernel over a different tree, no path reaches
      the emitter, so the image and the ray / hit counts equal plain final.txt's bit for bit
  G3  the double integrator on scenes/cornell.txt and on lit scenes with moving primitives (motion nodes): equal to
      the double oracle bit for bit on every scheduler; tile and sample shards sum to the whole image; rrtb_render_group
      over 2 contexts equals one
  G4  the float integrator on the same scenes: the same bits on every scheduler and shard, the usual float tolerance
      against the float oracle
  G5  rrtb_scene_set accepts type 3, rejects -1 and 4 and leaves the loaded scene renderable
  G6  staging a background then clearing it equals never staging one; the sky comes back on the next rrtb_scene_set;
      `rrt -i scenes/cornell.txt` writes a PNG and `rrt -G 2` the same bytes
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle_lib import Oracle
from rrt_b200.types import DIFFUSE_LIGHT, SceneArrays, material_dtype, sphere_dtype
from test_gpu_launch_space import POOL, S1, S2, SAMPLES, SIMPLE, TILES, _renders, _where, shard_paths
from test_lights import ANCHORS, CORNELL, as_fixed, check_two_level, emitter_only_scene, fixed, furnace_scene
from test_moving_instances import fast_spheres_scene, load, scene_text

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------
# G1: analytic anchors
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(ANCHORS))
@pytest.mark.parametrize("depth", [1, 2, 50])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_anchor_sums_on_the_gpu(ctx, name, depth, precision):
    build, miss, hit = ANCHORS[name]
    W, H, spp = 33, 17, 40
    scene = build(W, H)
    _, want, cnt = Oracle(scene).render_f64(W, H, spp, depth, S2)
    if depth == 1:
        hit = (0.0, 0.0, 0.0)  # the bounce off the small sphere would exceed the depth
    check_two_level(want, spp, miss, hit, (H // 2, W // 2), (0, 0))
    for label, img, st, count in _renders(ctx, scene, W, H, spp, depth, S2, precision, np.float64):
        got = as_fixed(img)
        assert got.tobytes() == want.tobytes(), (name, depth, label, _where(got, want))
        assert st["paths"] == W * H * spp
        if count:
            assert (st["rays"], st["hits"]) == (cnt["rays"], cnt["hits"]), (label, st, cnt)


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_anchor_clamp_on_the_gpu(ctx, precision):
    """Le = 3 at spp = 2^21 + 1 (per-sample clamp 2): every pixel sums to spp * fixed(2) = 2^62 + 2^41, read from the
    64-bit accumulator itself (beyond the double framebuffer's exact range)."""
    import torch

    W, H, spp = 2, 2, 2**21 + 1
    ctx.set_scene(emitter_only_scene(W, H, 3.0), use_bvh=True)
    for sched in (POOL, SIMPLE):
        acc = torch.zeros(3 * W * H, dtype=torch.int64, device="cuda")
        st = ctx.render_device(ctx.params(W, H, spp, 2, S1, 0, 1, TILES, True, sched, precision), acc.data_ptr())
        torch.cuda.synchronize()
        assert acc.cpu().numpy().tolist() == [spp * fixed(2.0)] * (3 * W * H), (precision, sched)
        assert st["rays"] == st["hits"] == W * H * spp


def test_scatter_hook_on_an_emitter(ctx):
    scene = furnace_scene(8, 4, 0.5)
    ctx.set_scene(scene)
    in16 = np.zeros((2, 16))
    in16[:, 3:6] = (0, 0, -1)
    in16[:, 10:13] = (0, 0, 1)
    in16[:, 13] = 1
    in16[:, 14] = (1, 0)
    rnd = (np.arange(8, dtype=np.uint64).reshape(2, 4) * 0x9E3779B9 % 2**32).astype(np.uint32)
    orc = Oracle(scene)
    got32, got64 = ctx.scatter(in16.astype(np.float32), rnd), ctx.scatter_f64(in16, rnd)
    assert got32[0].tolist() == got64[0].tolist() == [0, 0, 0, 0.75, 0.75, 0.75, 0, 0]
    assert got64.tobytes() == orc.scatter_f64(in16, rnd).tobytes()
    assert got32[:, 6].tolist() == [0, 1]


# ---------------------------------------------------------------------------------------------------------------
# G2: an emitter no path can reach
# ---------------------------------------------------------------------------------------------------------------
def buried_light(scene):
    """final.txt plus `material l diffuse_light 5 5 5` and a sphere of radius 1 at (0, -900, 0), deep inside the ground
    sphere: paths reach the ground's inside only through a rounding accident at a grazing bounce."""
    m = np.concatenate([scene.materials, np.array([(DIFFUSE_LIGHT, (5, 5, 5), 0)], material_dtype)])
    s = np.concatenate([scene.spheres, np.array([((0, -900, 0), 1.0, len(m) - 1)], sphere_dtype)])
    return SceneArrays(scene.camera, m, s, scene.mspheres, scene.triangles, scene.mtriangles)


def test_buried_light_is_not_reached_on_the_oracle():
    plain, _ = load_golden("final")
    lit = buried_light(plain)
    W, H, spp = 40, 27, 4
    for render in ("render", "render_f64"):
        a = getattr(Oracle(plain), render)(W, H, spp, 50, S1)
        b = getattr(Oracle(lit), render)(W, H, spp, 50, S1)
        assert a[1].tobytes() == b[1].tobytes() and (a[2]["rays"], a[2]["hits"]) == (b[2]["rays"], b[2]["hits"])


@pytest.mark.parametrize("W,H,spp", [(97, 61, 64), (400, 266, 8)])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_buried_light_image_equals_plain_final(ctx, W, H, spp, precision):
    plain, _ = load_golden("final")
    lit = buried_light(plain)
    dtype = np.float64 if precision == "f64" else np.float32
    a = _renders(ctx, plain, W, H, spp, 50, S1, precision, dtype)
    b = _renders(ctx, lit, W, H, spp, 50, S1, precision, dtype)
    for (label, img_a, st_a, count), (_, img_b, st_b, _) in zip(a, b):
        assert img_a.tobytes() == img_b.tobytes(), (label, _where(img_a, img_b))
        if count:
            assert (st_a["rays"], st_a["hits"]) == (st_b["rays"], st_b["hits"]), (label, st_a, st_b)


# ---------------------------------------------------------------------------------------------------------------
# G3 / G4: lit scenes, both integrators
# ---------------------------------------------------------------------------------------------------------------
def lit_fast_spheres():
    """64 fast moving spheres (motion nodes), a quarter of them emitters, under a dim background."""
    sc = fast_spheres_scene()
    m = np.concatenate([sc.materials, np.array([(DIFFUSE_LIGHT, (4.0, 3.0, 2.0), 0)], material_dtype)])
    ms = sc.mspheres.copy()
    ms["material"][::4] = len(m) - 1
    return SceneArrays(sc.camera, m, sc.spheres, ms, sc.triangles, background=(0.05, 0.06, 0.1))


LIT_MTRI = "material lamp diffuse_light 3 3 2.5\nsphere 0.4 1.6 -0.4 0.35 lamp\nbackground 0.1 0.1 0.15\n"


@pytest.fixture(scope="module")
def lit_scenes(tmp_path_factory, built_lib):
    from rrt_b200 import Scene

    d = tmp_path_factory.mktemp("lights")
    out = {"cornell": Scene.from_file(CORNELL, 61, 45).arrays, "fast": lit_fast_spheres()}
    out["mtri"] = load(d, scene_text("moving") + LIT_MTRI, name="mtri.txt").arrays  # 8 moving triangles, open shutter
    assert len(out["mtri"].mtriangles) == 8 and out["mtri"].background is not None
    return out


LIT_CASES = [("cornell", 61, 45, 24, 50), ("cornell", 33, 17, 7, 3), ("fast", 61, 45, 16, 50), ("mtri", 61, 45, 16, 50)]


@pytest.mark.parametrize("case", LIT_CASES, ids=lambda c: "%s-%dx%d-s%d-d%d" % c)
def test_f64_lit_render_equals_oracle(ctx, lit_scenes, case):
    name, W, H, spp, depth = case
    scene = lit_scenes[name]
    want, _, cnt = Oracle(scene).render_f64(W, H, spp, depth, S2)
    for label, img, st, count in _renders(ctx, scene, W, H, spp, depth, S2, "f64", np.float64):
        assert img.tobytes() == want.tobytes(), (case, label, _where(img, want))
        if count:
            assert (st["rays"], st["hits"]) == (cnt["rays"], cnt["hits"]), (case, label, st, cnt)


@pytest.mark.parametrize("case", LIT_CASES, ids=lambda c: "%s-%dx%d-s%d-d%d" % c)
def test_f32_lit_render_same_bits_on_every_scheduler(ctx, lit_scenes, case):
    name, W, H, spp, depth = case
    scene = lit_scenes[name]
    runs = _renders(ctx, scene, W, H, spp, depth, S2, "f32", np.float32)
    first = runs[0][1]
    for label, img, st, count in runs:
        assert img.tobytes() == first.tobytes(), (case, label, _where(img, first))
    assert len({(st["rays"], st["hits"]) for _, _, st, count in runs if count}) == 1
    ref, _, _ = Oracle(scene).render(W, H, spp, depth, S2)
    a = np.sqrt(first.astype(np.float64) / spp).clip(0, 1)
    b = np.sqrt(ref.astype(np.float64) / spp).clip(0, 1)
    close = np.abs(a - b).max(axis=2) < 1e-3
    assert close.mean() > 0.97, (case, close.mean())
    assert abs(a.mean() - b.mean()) < 2e-3, (case, a.mean(), b.mean())


@pytest.mark.parametrize("name", ["cornell", "fast", "mtri"])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_lit_shards_sum_to_the_whole_image(ctx, lit_scenes, name, precision):
    scene = lit_scenes[name]
    W, H, spp = 33, 17, 6
    for sched in (POOL, SIMPLE):
        ctx.set_scene(scene, use_bvh=True)
        whole, _ = ctx.render(W, H, spp, 50, seed=S1, scheduler=sched, dtype=np.float64, precision=precision)
        for world in (2, 3):
            for mode in (TILES, SAMPLES):
                acc = np.zeros_like(whole)
                for rank in range(world):
                    part, st = ctx.render(W, H, spp, 50, seed=S1, rank=rank, world=world, shard_mode=mode, scheduler=sched,
                                          dtype=np.float64, precision=precision)
                    paths, own = shard_paths(W, H, spp, rank, world, mode)
                    assert st["paths"] == paths and not part[~own].any()
                    acc += part
                assert acc.tobytes() == whole.tobytes(), (name, sched, world, mode, _where(acc, whole))


@pytest.mark.parametrize("name", ["cornell", "fast"])
def test_lit_render_group_equals_one_context(lit_scenes, name):
    from rrt_b200 import Context, render_group

    scene = lit_scenes[name]
    W, H, spp = 61, 45, 8
    ctxs = [Context(0), Context(0)]
    try:
        for c in ctxs:
            c.set_scene(scene, use_bvh=True)
        for precision, dtype in (("f32", np.float32), ("f64", np.float64)):
            want, _ = ctxs[0].render(W, H, spp, 50, seed=S1, dtype=dtype, precision=precision)
            for mode in (TILES, SAMPLES):
                got, _ = render_group(ctxs, W, H, spp, 50, seed=S1, shard_mode=mode, dtype=dtype, precision=precision)
                assert got.tobytes() == want.tobytes(), (name, precision, mode)
    finally:
        for c in ctxs:
            c.close()


# ---------------------------------------------------------------------------------------------------------------
# G5 / G6: the C ABI
# ---------------------------------------------------------------------------------------------------------------
def _scene_set(ctx, a, use_bvh=True):
    """rrtb_scene_set alone: whatever is staged on the context is consumed, nothing new is staged"""
    vp = lambda x: C.c_void_p(x.ctypes.data) if x.size else C.c_void_p(0)
    return ctx.lib.rrtb_scene_set(ctx.h, vp(a.camera), vp(a.materials), len(a.materials), vp(a.spheres), len(a.spheres),
                                  vp(a.mspheres), len(a.mspheres), vp(a.triangles), len(a.triangles), 1 if use_bvh else 0)


def test_scene_set_material_types(ctx):
    from rrt_b200 import RrtbError

    scene = furnace_scene(16, 8, 0.5)
    ctx.set_scene(scene)
    want, _ = ctx.render(16, 8, 4, 50, dtype=np.float64, precision="f64")
    for t in (-1, 4):
        bad = SceneArrays(scene.camera, scene.materials.copy(), scene.spheres)
        bad.materials["type"][1] = t
        with pytest.raises(RrtbError) as e:
            ctx.set_scene(bad)
        assert e.value.status == -1, t  # RRTB_ERR_INVALID
        got, _ = ctx.render(16, 8, 4, 50, dtype=np.float64, precision="f64")
        assert got.tobytes() == want.tobytes(), t  # the loaded scene still renders, with its emitter
    assert want[4, 0].tolist() == [4 * 0.75] * 3


def test_staging_then_clearing_a_background_is_no_background(ctx):
    plain, _ = load_golden("test2")
    W, H, spp = 64, 40, 8
    bg = np.array([0.25, 0.5, 1.0], np.float32)
    st = ctx.lib.rrtb_scene_stage_background
    ctx.set_scene(plain)
    sky, _ = ctx.render(W, H, spp, 50, seed=S1, dtype=np.float64, precision="f64")
    assert st(ctx.h, C.c_void_p(bg.ctypes.data)) == 0 and st(ctx.h, None) == 0
    assert _scene_set(ctx, plain) == 0
    got, _ = ctx.render(W, H, spp, 50, seed=S1, dtype=np.float64, precision="f64")
    assert got.tobytes() == sky.tobytes()
    # staged: the background replaces the sky (the oracle agrees bit for bit) ...
    assert st(ctx.h, C.c_void_p(bg.ctypes.data)) == 0 and _scene_set(ctx, plain) == 0
    with_bg, _ = ctx.render(W, H, spp, 50, seed=S1, dtype=np.float64, precision="f64")
    want, _, _ = Oracle(SceneArrays(plain.camera, plain.materials, plain.spheres, plain.mspheres, plain.triangles,
                                 background=bg)).render_f64(W, H, spp, 50, S1)
    assert with_bg.tobytes() == want.tobytes() and with_bg.tobytes() != sky.tobytes()
    # ... and is consumed: the next rrtb_scene_set without a staging call has the sky again
    assert _scene_set(ctx, plain) == 0
    again, _ = ctx.render(W, H, spp, 50, seed=S1, dtype=np.float64, precision="f64")
    assert again.tobytes() == sky.tobytes()


def test_cli_renders_cornell(tmp_path, built_lib):
    from PIL import Image

    exe = os.path.join(ROOT, "rrt_b200", "bin", "rrt")
    args = [exe, "-i", CORNELL, "-w", "120", "-h", "120", "-s", "16"]
    outs = []
    for g in (1, 2):
        out = tmp_path / ("g%d.png" % g)
        r = subprocess.run(args + ["-G", str(g), "-o", str(out)], capture_output=True, text=True, timeout=600,
                           env=dict(os.environ, RRTB_GROUP_SAME_DEVICE="1"))
        assert r.returncode == 0, r.stderr
        outs.append(out.read_bytes())
    assert outs[0] == outs[1]
    img = np.asarray(Image.open(tmp_path / "g1.png"))
    assert img.shape == (120, 120, 3) and img.max() == 255 and img.mean() > 20  # the light is seen, the room is lit
