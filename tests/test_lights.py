"""-m "not gpu": diffuse_light emitters and a constant background (include/rrtb.h RRTB_DIFFUSE_LIGHT,
rrtb_scene_stage_background): the scene grammar, the Python scene arrays and the analytic anchors on both CPU oracles (with the lights terms of
tests/oracle_lights, see tests/lights_oracle.py).

The anchors are scenes in which every camera path ends after at most two segments with a radiance that is one product
of exactly representable values, so each pixel sum is known exactly:

  furnace     the camera inside an emitting sphere (Le = 0.75) that holds one convex lambertian sphere of albedo a: a
              path sees the emitter (0.75) or the sphere, whose bounce leaves it and reaches the emitter (a * 0.75)
  background  one lambertian sphere of albedo a under a constant background B: a miss is B, a hit a * B
  clamp       the camera inside an emitter of Le = 3 at 2^21 < spp <= 2^22, where the per-sample clamp C is 2

tests/test_gpu_lights.py renders the same scenes on the GPU and expects the same sums.
"""
import os

import numpy as np
import pytest

from conftest import ROOT, load_golden
from lights_oracle import LitOracle
from oracle_lib import Oracle, camera_derive, ref_scene_path
from rrt_b200.types import DIFFUSE_LIGHT, SceneArrays, material_dtype, sphere_dtype

CORNELL = os.path.join(ROOT, "scenes", "cornell.txt")
CAM = "camera 0 2 5  0 0 -1  0 1 0  30 0.1 6\n"
MAT = "material m lambertian 0.5 0.5 0.5\n"


def fixed(x):
    """x * 2^40 for an x exactly representable in float (the pixel sums' fixed point)"""
    v = float(np.float32(x)) * 2.0**40
    assert v == int(v)
    return int(v)


# ---------------------------------------------------------------------------------------------------------------
# analytic scenes (also used by tests/test_gpu_lights.py)
# ---------------------------------------------------------------------------------------------------------------
def _scene(W, H, mats, spheres, background=None):
    m = np.zeros(len(mats), material_dtype)
    for k, (t, alb) in enumerate(mats):
        m[k]["type"], m[k]["albedo"] = t, alb
    s = np.zeros(len(spheres), sphere_dtype)
    for k, (c, r, mat) in enumerate(spheres):
        s[k] = (c, r, mat)
    cam = camera_derive((0, 0, 0), (0, 0, -1), (0, 1, 0), 40.0, W / H, 0.0, 1.0)
    return SceneArrays(cam, m, s, background=background)


def furnace_scene(W, H, albedo, le=0.75):
    """The camera inside an emitter of radius 10 around the origin; a lambertian sphere of radius 1 at distance 3."""
    return _scene(W, H, [(0, (albedo,) * 3), (DIFFUSE_LIGHT, (le,) * 3)], [((0, 0, 0), 10.0, 1), ((0, 0, -3), 1.0, 0)])


def background_scene(W, H, albedo, bg):
    return _scene(W, H, [(0, (albedo,) * 3)], [((0, 0, -3), 1.0, 0)], background=bg)


def emitter_only_scene(W, H, le):
    return _scene(W, H, [(DIFFUSE_LIGHT, (le,) * 3)], [((0, 0, 0), 10.0, 0)])


# (scene builder, radiance of a path that misses the small sphere, of one that hits it), per channel
ANCHORS = {
    "furnace-a1": (lambda W, H: furnace_scene(W, H, 1.0), (0.75,) * 3, (0.75,) * 3),
    "furnace-a0.5": (lambda W, H: furnace_scene(W, H, 0.5), (0.75,) * 3, (0.375,) * 3),
    "background-a0.5": (lambda W, H: background_scene(W, H, 0.5, (0.25, 0.5, 0.75)), (0.25, 0.5, 0.75), (0.125, 0.25, 0.375)),
}


def check_two_level(sums, spp, miss, hit, center, corner):
    """Every pixel is k samples of `hit` and spp - k of `miss`, the same k in every channel; the centre pixel is all
    hit and the corner pixel all miss.  `sums` are the 2^40 fixed-point sums, [H, W, 3] integers."""
    sums = np.asarray(sums, dtype=object)
    lo, hi = [fixed(x) for x in miss], [fixed(x) for x in hit]
    H, W, _ = sums.shape
    ks = np.zeros((H, W), np.int64)
    for j in range(H):
        for i in range(W):
            k = None
            for c in range(3):
                v = int(sums[j, i, c]) - spp * lo[c]
                if hi[c] == lo[c]:
                    assert v == 0, (j, i, c)
                    continue
                assert v % (hi[c] - lo[c]) == 0, (j, i, c, int(sums[j, i, c]))
                kc = v // (hi[c] - lo[c])
                assert 0 <= kc <= spp and (k is None or kc == k), (j, i, c, kc, k)
                k = kc
            ks[j, i] = spp if k is None else k
    for (j, i), want in ((center, hi), (corner, lo)):
        assert [int(sums[j, i, c]) for c in range(3)] == [spp * x for x in want], ((j, i), sums[j, i])
    return ks


def as_fixed(img64):
    """The double framebuffer times 2^40: the fixed-point sums, exact while they stay below 2^53."""
    v = np.asarray(img64, np.float64) * 2.0**40
    assert np.all(v < 2.0**53) and np.all(v == np.floor(v))
    return v.astype(np.uint64)


# ---------------------------------------------------------------------------------------------------------------
# C1: scene grammar
# ---------------------------------------------------------------------------------------------------------------
def _write(tmp_path, text, name="s.txt"):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def test_parser_diffuse_light(tmp_path, built_lib):
    from rrt_b200 import Scene

    s = Scene.from_file(_write(tmp_path, CAM + MAT + "material lamp diffuse_light 4 2.5 -1\nsphere 0 0 0 1 lamp\n"), 120, 80)
    m = s.arrays.materials
    assert m["type"].tolist() == [0, DIFFUSE_LIGHT]
    assert m["albedo"][1].tolist() == [4.0, 2.5, -1.0] and m["param"][1] == 0.0  # Le, unvalidated (a negative one adds 0)
    assert s.arrays.spheres["material"].tolist() == [1]
    assert s.arrays.background is None


def test_parser_background(tmp_path, built_lib):
    from rrt_b200 import Scene, SceneError

    text = CAM + "background 0.5 0.25 2\n" + MAT + "sphere 0 0 0 1 m\nbackground 0.125 0 1\n"
    a = Scene.from_file(_write(tmp_path, text), 120, 80).arrays
    assert a.background.dtype == np.float32 and a.background.tolist() == [0.125, 0.0, 1.0]  # the last line wins
    without = Scene.from_file(_write(tmp_path, CAM + MAT + "sphere 0 0 0 1 m\n", "b.txt"), 120, 80).arrays
    assert without.background is None
    for k in ("camera", "materials", "spheres"):  # a background changes nothing else
        assert getattr(a, k).tobytes() == getattr(without, k).tobytes()
    # a short line fails as a short sphere line does: a missing number is a bad number (exit code 1)
    with pytest.raises(SceneError) as e:
        Scene.from_file(_write(tmp_path, CAM + MAT + "sphere 0 0 0 1 m\nbackground 0.5 0.5\n", "c.txt"), 120, 80)
    assert e.value.ref_exit_code == 1
    with pytest.raises(SceneError) as e:
        Scene.from_file(_write(tmp_path, CAM + MAT + "sphere 0 0 0\n", "d.txt"), 120, 80)
    assert e.value.ref_exit_code == 1


def test_parser_still_rejects_other_material_types(tmp_path, built_lib):
    from rrt_b200 import Scene, SceneError

    for t in ("plastic 1 1 1", "diffuse 1 1 1", "light 1 1 1", "diffuse_lights 1 1 1"):
        with pytest.raises(SceneError) as e:
            Scene.from_file(_write(tmp_path, CAM + "material m %s\nsphere 0 0 0 1 m\n" % t), 120, 80)
        assert e.value.ref_exit_code == 3, t


@pytest.mark.parametrize("name", ["test1", "test2", "test3", "final"])
def test_shipped_scenes_parse_as_before(name, built_lib):
    """The stand-ins of the reference's scenes have neither lights nor a background: the same arrays as the fixture."""
    from rrt_b200 import Scene

    p = ref_scene_path(name + ".txt")
    if not p:
        pytest.skip("scene text not staged")
    gold, d = load_golden(name)
    s = Scene.from_file(p, int(d["W"]), int(d["H"]))
    for k in ("camera", "materials", "spheres", "mspheres", "triangles", "mtriangles"):
        assert getattr(s.arrays, k).tobytes() == getattr(gold, k).tobytes(), (name, k)
    assert s.arrays.background is None and gold.background is None
    assert DIFFUSE_LIGHT not in s.arrays.materials["type"]


def test_cornell_scene(built_lib):
    from rrt_b200 import Scene

    s = Scene.from_file(CORNELL, 400, 400)
    a = s.arrays
    assert a.background.tolist() == [0.0, 0.0, 0.0]
    assert a.materials["type"].tolist() == [0, 0, 0, DIFFUSE_LIGHT, 1, 2]
    assert a.materials["albedo"][3].tolist() == [15.0] * 3
    assert len(a.spheres) == 2 and len(a.triangles) == 12 and s.n_objs == 3 and s.n_obj_insts == 6
    light = a.triangles[a.triangles["material"] == 3]
    assert len(light) == 2 and np.all(light["v0"][:, 1] == 554) and np.all(light["v1"][:, 1] == 554)


# ---------------------------------------------------------------------------------------------------------------
# Python scene arrays
# ---------------------------------------------------------------------------------------------------------------
def test_scene_arrays_carry_the_background():
    sc = background_scene(8, 4, 0.5, (0.25, 0.5, 0.75))
    d = sc.to_npz_dict()
    assert d["background"].tolist() == [0.25, 0.5, 0.75]
    back = SceneArrays.from_npz_dict(d)
    assert back.background.tolist() == [0.25, 0.5, 0.75] and back.background.dtype == np.float32
    sky = SceneArrays(sc.camera, sc.materials, sc.spheres)
    assert "background" not in sky.to_npz_dict() and SceneArrays.from_npz_dict(sky.to_npz_dict()).background is None
    old, _ = load_golden("final")  # fixtures written before the field existed
    assert old.background is None


# ---------------------------------------------------------------------------------------------------------------
# C2: analytic anchors on both oracles
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(ANCHORS))
@pytest.mark.parametrize("depth", [2, 50])
def test_anchor_sums_on_the_oracles(name, depth):
    build, miss, hit = ANCHORS[name]
    W, H, spp = 9, 7, 24
    scene = build(W, H)
    orc = LitOracle(scene)
    ks = []
    for bvh in (True, False):
        _, f32, c32 = orc.render(W, H, spp, depth, 1984, use_bvh=bvh)
        _, f64, c64 = orc.render_f64(W, H, spp, depth, 1984, use_bvh=bvh)
        assert f32.tobytes() == f64.tobytes()  # one exact product per sample: both integrators agree bit for bit
        ks.append(check_two_level(f32, spp, miss, hit, (H // 2, W // 2), (0, 0)))
        # every path: the camera segment, and a second one for the paths that hit the small sphere
        n_hit = c64["rays"] - W * H * spp
        assert c64["paths"] == W * H * spp and 0 < n_hit < W * H * spp
        assert c32["rays"] == c64["rays"] and c32["hits"] == c64["hits"]
        assert c64["hits"] == (c64["rays"] if name.startswith("furnace") else n_hit)
        if hit != miss:  # the sums tell how many samples of each pixel hit the sphere
            assert ks[-1].sum() == n_hit
    assert np.array_equal(ks[0], ks[1])


@pytest.mark.parametrize("name", sorted(ANCHORS))
def test_anchor_at_depth_one(name):
    """One segment per path: a hit on the small sphere is black (its bounce would exceed the depth); the emitter and the
    background still count."""
    build, miss, _ = ANCHORS[name]
    W, H, spp = 9, 7, 8
    _, f, _ = LitOracle(build(W, H)).render_f64(W, H, spp, 1, 1984)
    check_two_level(f, spp, miss, (0.0, 0.0, 0.0), (H // 2, W // 2), (0, 0))


def test_anchor_clamp_on_the_oracle():
    """Le = 3 at spp = 2^21 + 1, where the per-sample clamp is 2: every pixel sums to exactly spp * fixed(2)."""
    W, H, spp = 2, 2, 2**21 + 1
    _, f, _ = LitOracle(emitter_only_scene(W, H, 3.0)).render_f64(W, H, spp, 2, 1984, use_bvh=False)
    assert np.all(f == spp * fixed(2.0))


def test_scatter_reports_no_scatter_for_an_emitter():
    scene = furnace_scene(8, 4, 0.5)
    orc = LitOracle(scene)
    in16 = np.zeros((2, 16))
    in16[:, 3:6] = (0, 0, -1)
    in16[:, 10:13] = (0, 0, 1)
    in16[:, 13] = 1
    in16[:, 14] = (1, 0)  # the emitter, then the lambertian
    rnd = np.arange(8, dtype=np.uint32).reshape(2, 4) * 0x9E3779B9
    for out in (orc.scatter(in16, rnd), orc.scatter_f64(in16, rnd)):
        assert out[0].tolist() == [0, 0, 0, 0.75, 0.75, 0.75, 0, 0]
        assert out[1, 6] == 1 and out[1, 3] == 0.5


@pytest.mark.parametrize("name", ["test2", "final"])
def test_lights_oracle_without_lights_is_the_oracle(name):
    """The oracle with lights, on a scene with neither emitter nor background, is the plain oracle bit for bit."""
    scene, _ = load_golden(name)
    W, H, spp = 24, 16, 3
    a, b = Oracle(scene), LitOracle(scene)
    for bvh in (True, False):
        for r in ("render", "render_f64"):
            x, y = getattr(a, r)(W, H, spp, 50, 7, use_bvh=bvh), getattr(b, r)(W, H, spp, 50, 7, use_bvh=bvh)
            assert x[1].tobytes() == y[1].tobytes() and x[2] == y[2], (name, r, bvh)
    x, y = a.render(W, H, spp, 50, 7, rank=1, world=3, shard_mode=0), b.render(W, H, spp, 50, 7, rank=1, world=3, shard_mode=0)
    assert x[1].tobytes() == y[1].tobytes()
    rng = np.random.default_rng(3)
    in16 = rng.normal(size=(64, 16))
    in16[:, 13] = rng.integers(0, 2, 64)
    in16[:, 14] = rng.integers(0, len(scene.materials), 64)
    rnd = rng.integers(0, 2**32, size=(64, 4), dtype=np.uint32)
    assert a.scatter(in16, rnd).tobytes() == b.scatter(in16, rnd).tobytes()
    assert a.scatter_f64(in16, rnd).tobytes() == b.scatter_f64(in16, rnd).tobytes()
