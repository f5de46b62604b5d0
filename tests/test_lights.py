"""-m "not gpu": diffuse_light emitters and a constant background (include/rrtb.h RRTB_DIFFUSE_LIGHT,
rrtb_scene_stage_background): the scene grammar, the Python scene arrays, the analytic anchors on both integrators of
the CPU oracle (which carries the emitted and background terms itself, oracle/rrt_oracle.h), and the oracle's outputs
pinned by digest on scenes with and without lights.

The anchors are scenes in which every camera path ends after at most two segments with a radiance that is one product
of exactly representable values, so each pixel sum is known exactly:

  furnace     the camera inside an emitting sphere (Le = 0.75) that holds one convex lambertian sphere of albedo a: a
              path sees the emitter (0.75) or the sphere, whose bounce leaves it and reaches the emitter (a * 0.75)
  background  one lambertian sphere of albedo a under a constant background B: a miss is B, a hit a * B
  clamp       the camera inside an emitter of Le = 3 at 2^21 < spp <= 2^22, where the per-sample clamp C is 2

tests/test_gpu_lights.py renders the same scenes on the GPU and expects the same sums.
"""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import ROOT, load_golden
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
# C2: analytic anchors on both integrators of the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(ANCHORS))
@pytest.mark.parametrize("depth", [2, 50])
def test_anchor_sums_on_the_oracles(name, depth):
    build, miss, hit = ANCHORS[name]
    W, H, spp = 9, 7, 24
    scene = build(W, H)
    orc = Oracle(scene)
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
    _, f, _ = Oracle(build(W, H)).render_f64(W, H, spp, 1, 1984)
    check_two_level(f, spp, miss, (0.0, 0.0, 0.0), (H // 2, W // 2), (0, 0))


def test_anchor_clamp_on_the_oracle():
    """Le = 3 at spp = 2^21 + 1, where the per-sample clamp is 2: every pixel sums to exactly spp * fixed(2)."""
    W, H, spp = 2, 2, 2**21 + 1
    _, f, _ = Oracle(emitter_only_scene(W, H, 3.0)).render_f64(W, H, spp, 2, 1984, use_bvh=False)
    assert np.all(f == spp * fixed(2.0))


def test_scatter_reports_no_scatter_for_an_emitter():
    scene = furnace_scene(8, 4, 0.5)
    orc = Oracle(scene)
    in16 = np.zeros((2, 16))
    in16[:, 3:6] = (0, 0, -1)
    in16[:, 10:13] = (0, 0, 1)
    in16[:, 13] = 1
    in16[:, 14] = (1, 0)  # the emitter, then the lambertian
    rnd = np.arange(8, dtype=np.uint32).reshape(2, 4) * 0x9E3779B9
    for out in (orc.scatter(in16, rnd), orc.scatter_f64(in16, rnd)):
        assert out[0].tolist() == [0, 0, 0, 0.75, 0.75, 0.75, 0, 0]
        assert out[1, 6] == 1 and out[1, 3] == 0.5


# ---------------------------------------------------------------------------------------------------------------
# C3: the oracle pinned on the CPU
# ---------------------------------------------------------------------------------------------------------------
PIN_W, PIN_H, PIN_SPP, PIN_DEPTH, PIN_SEED = 24, 16, 3, 50, 7

# scene -> output -> SHA-256, made as test_oracle_outputs_are_pinned says; data, never to be regenerated by a refactor
ORACLE_PINS = {
    "test2": {
        "render/bvh": "bfc47d425042f12b7d4ebb69d9fd6c1ded3f4c897e1e3020e390b9f4366d94db",
        "render/scan": "93f80c91ee11d2ae31a5b99a0a1f34203078663771a71d8512fe55d5c35cadaa",
        "render_f64/bvh": "f593ae3f4db6cd1d5ee1ca732b6594bf49f8873fbcf45264378278fc32ce20a2",
        "render_f64/scan": "f593ae3f4db6cd1d5ee1ca732b6594bf49f8873fbcf45264378278fc32ce20a2",
        "render/bvh/tile-1-of-3": "8b02411963e23111b2199a6b64fd25ede52860011e04442e2448e6be07d1729d",
        "scatter": "aa22ae5d77459119d58754d864c6e08cc4617c79e9fc0a6db66a3303414a09d0",
        "scatter_f64": "28b219b76ca42fcfcbbd3692cc4f7ca1aea7c94199544d2dc275df9fdb25f6e4",
    },
    "test3": {
        "render/bvh": "1fd29dc0f7355fed87a691584e3c65d4550c20772876479a56e5d6412cf612b2",
        "render/scan": "ca0eef29999db1029a5471e0230c2242f8451d9cd1d075c0a3e6961c73b9050b",
        "render_f64/bvh": "5f85663e74e1d4d6452135663796ccac253e47b914e94a986689ebdcb3c3394d",
        "render_f64/scan": "5f85663e74e1d4d6452135663796ccac253e47b914e94a986689ebdcb3c3394d",
        "render/bvh/tile-1-of-3": "8d8efa896c948b6922192bc11aa7c79dfe4b42b00010057d43ee5f99c860115a",
        "scatter": "a51d7c13f3651d972ace5d1e3b431900d82c5a601fadca46a811a22a72cefe80",
        "scatter_f64": "3832a0526a294e25f16cc414aea71b5d2c02170bd63dcbc44cb0ff19e49d315b",
    },
    "final": {
        "render/bvh": "7cd9a96279f70a997114a625c32667e891e18000ea96b855c69db55b2c369532",
        "render/scan": "d5fd04771898a1fb4fd1fc111340c9f4c725900e0d25a517a9f13d91eb265f6e",
        "render_f64/bvh": "ee524c3d6eb62095d38fdf56f2f1fb6d7c51ca4f904885f6b64da98de3dcfbff",
        "render_f64/scan": "ee524c3d6eb62095d38fdf56f2f1fb6d7c51ca4f904885f6b64da98de3dcfbff",
        "render/bvh/tile-1-of-3": "17933ca73ac0ab18cf715fe15aecd2b940e04128269b6a9236ca30664502d853",
        "scatter": "375ae995875b777629ca807d2c25684ac3cb77eea62bf158bc06fa743527a7b7",
        "scatter_f64": "7be9360b108167358168584f779fb8b05cf267e49ad1663d665f28fabc51c30e",
    },
    "background-a0.5": {
        "render/bvh": "fbc1f6124b49706bf5a254d361cffbdb629afe9fdcfbf84c78aa618aac553670",
        "render/scan": "b1f11552ef88672d2d351752efd957e8dbb3675fb03be26caf1ebe2cf2840d5b",
        "render_f64/bvh": "fbc1f6124b49706bf5a254d361cffbdb629afe9fdcfbf84c78aa618aac553670",
        "render_f64/scan": "fbc1f6124b49706bf5a254d361cffbdb629afe9fdcfbf84c78aa618aac553670",
        "render/bvh/tile-1-of-3": "707b626a2a2fd133ad3a339002f627babd5ac0521f4637488c4c6017ece2df50",
        "scatter": "75ed123957470cbe767b5cc047e5a3c59ac1cb67eb15302f82aca3c1ec2d64c5",
        "scatter_f64": "2b94de0780a434e0309549f155260a9d539c38435aff717601158e6cf26e11e6",
    },
    "furnace-a0.5": {
        "render/bvh": "78d196de3a7af7c6956535061b33401b3993bb12a0f8bd50cfc5889562de6902",
        "render/scan": "6fd1e86cf82ae31988877020e72a949b9aae662e7e32c6b300bfbb929ed49474",
        "render_f64/bvh": "c6e38d70929efc5a52f943938563c194abbc0cac05263d31688003ed196937a1",
        "render_f64/scan": "c6e38d70929efc5a52f943938563c194abbc0cac05263d31688003ed196937a1",
        "render/bvh/tile-1-of-3": "d228c379331595516f0e6b9a952b40eeda3ab4d0337106a4049a3fcc949b33c5",
        "scatter": "f52c92afaa7007e77012bed647769c5189f618e231df5eb4c05a3f72baf5eda9",
        "scatter_f64": "96acc1b7214d14167e6550d1cfce7372d2660271b16cbe5e31b8bcecce3293d7",
    },
    "furnace-a1": {
        "render/bvh": "2c9ea54073d34a00586dd755089980a1727eaafcab66883523661743d923a354",
        "render/scan": "f9c474aea6c0cb420cd9fdb4d6bd60359da9f7a4f51f07124081c58b957f4343",
        "render_f64/bvh": "5b1dca39025261a1d644413f63c9d0deb9f365c8bd4b46c10cad453ace53dc33",
        "render_f64/scan": "5b1dca39025261a1d644413f63c9d0deb9f365c8bd4b46c10cad453ace53dc33",
        "render/bvh/tile-1-of-3": "b6ad88903160dcfe0ce883b97788f8b9cc2337fd9c26a35da0fed9b89606631f",
        "scatter": "a90e2fdf22404d607c323ec66eaee0e157a0f627dbaf3e8d5eb39dbeefbb6ba9",
        "scatter_f64": "f7b5ccbcd0a231e0ec993593b7ef029c4c07e725e7eef49aaa35369ffaf18a38",
    },
    "cornell": {
        "render/bvh": "c580a9ae82c8eb3a213f555f76da3c79ae0801eabb774c0f374f145ad2842d48",
        "render/scan": "90ad2ca0b7528ef68ece1cdac58a656d86fae5848459083a45d36d95bd1bc1b4",
        "render_f64/bvh": "5f45fff9b36eb1fe22cf3b0285f972e32376a3e69501819964fa2c8157f19795",
        "render_f64/scan": "5f45fff9b36eb1fe22cf3b0285f972e32376a3e69501819964fa2c8157f19795",
        "render/bvh/tile-1-of-3": "23e2c03aa83d36d2bcb2be3d59bf5a07880fdd39d4bc5dd9dc2eac5c76e50be8",
        "scatter": "fa3fa8029797c2b2be6eb5bf2188bf0b30b7ccb90e809e9f3e92e4e65bbbab55",
        "scatter_f64": "b8cdd165ef4a54922a7ad3b504a2bc2b1c7be3bdd504141897b18d78fca27f4f",
    },
}


def pin_scene(name):
    """A scene of ORACLE_PINS at PIN_W x PIN_H: a golden fixture, an anchor or scenes/cornell.txt (needs the library)"""
    if name == "cornell":
        from rrt_b200 import Scene

        return Scene.from_file(CORNELL, PIN_W, PIN_H).arrays
    if name in ANCHORS:
        return ANCHORS[name][0](PIN_W, PIN_H)
    return load_golden(name)[0]


def oracle_digests(orc):
    """SHA-256 of each pinned output of an oracle bound to a scene: a render's fixed-point framebuffer followed by its
    counters (JSON, sorted keys); a scatter hook's output array on 64 seeded random inputs over all of the scene's
    materials"""
    sha = lambda *parts: hashlib.sha256(b"".join(parts)).hexdigest()
    W, H, spp, depth, seed = PIN_W, PIN_H, PIN_SPP, PIN_DEPTH, PIN_SEED
    out = {}
    for r in ("render", "render_f64"):
        for bvh in (True, False):
            _, f, cnt = getattr(orc, r)(W, H, spp, depth, seed, use_bvh=bvh)
            out["%s/%s" % (r, "bvh" if bvh else "scan")] = sha(f.tobytes(), json.dumps(cnt, sort_keys=True).encode())
    _, f, cnt = orc.render(W, H, spp, depth, seed, rank=1, world=3, shard_mode=0)  # RRTB_SHARD_TILES
    out["render/bvh/tile-1-of-3"] = sha(f.tobytes(), json.dumps(cnt, sort_keys=True).encode())
    rng = np.random.default_rng(3)
    in16 = rng.normal(size=(64, 16))
    in16[:, 13] = rng.integers(0, 2, 64)
    in16[:, 14] = rng.integers(0, len(orc.scene.materials), 64)
    rnd = rng.integers(0, 2**32, size=(64, 4), dtype=np.uint32)
    out["scatter"] = sha(orc.scatter(in16, rnd).tobytes())
    out["scatter_f64"] = sha(orc.scatter_f64(in16, rnd).tobytes())
    return out


@pytest.mark.parametrize("name", list(ORACLE_PINS))
def test_oracle_outputs_are_pinned(name, request):
    """The oracle's framebuffers, counters and scatter outputs equal the digests of ORACLE_PINS: both integrators through
    the LBVH and the flat scan, a tile shard and both scatter hooks, on test2, test3 and final (no lights), on the three
    anchors and on cornell.txt (emitters, a background).

    The digests were computed once with oracle_digests at commit d7e664a, the last one with a separate oracle for
    lights: its plain oracle for test2, test3 and final, its oracle with lights for the others.  The oracle is what the
    GPU is held to bit for bit and the only check of the lights on a machine without a GPU, so a refactor of it must
    leave every digest as it is.  Only a change of what a path computes may change this table, in the same change as
    the GPU integrators."""
    if name == "cornell":
        request.getfixturevalue("built_lib")
    got = oracle_digests(Oracle(pin_scene(name)))
    assert got == ORACLE_PINS[name], [k for k in got if got[k] != ORACLE_PINS[name][k]]
