"""-m "not gpu": the first-hit AOVs (include/rrtb.h rrtb_render_aov) on the CPU oracle -- analytic anchors, tree /
scan and shard consistency, pinned outputs -- and the PFM writer and the `-A` usage errors of the drop-in."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle_lib import ORACLE_DIR, Oracle, build_oracle, camera_derive, oracle_lib
from rrt_b200.types import DIELECTRIC, DIFFUSE_LIGHT, LAMBERTIAN, SceneArrays, material_dtype, sphere_dtype, triangle_dtype

EXE = os.path.join(ROOT, "rrt_b200", "bin", "rrt")
CORNELL = os.path.join(ROOT, "scenes", "cornell.txt")
PRECISIONS = ("f32", "f64")
D = 5.0  # distance of the plane from the camera


# ---------------------------------------------------------------------------------------------------------------
# analytic scenes (also used by tests/test_gpu_aov.py)
# ---------------------------------------------------------------------------------------------------------------
def plane_scene(W, H, mtype=LAMBERTIAN, albedo=(0.2, 0.4, 0.6), z=-D, look=-1.0):
    """Two triangles forming the plane at `z`, perpendicular to a pinhole camera at the origin that looks along
    (0, 0, look) and sees nothing but the plane (look = -1) or nothing at all (look = +1 with z < 0)."""
    m = np.zeros(1, material_dtype)
    m[0]["type"], m[0]["albedo"], m[0]["param"] = mtype, albedo, 1.5
    t = np.zeros(2, triangle_dtype)
    a, b, c, d = (-100, -100, z), (100, -100, z), (100, 100, z), (-100, 100, z)
    t[0] = (a, b, c, 0)
    t[1] = (a, c, d, 0)
    cam = camera_derive((0, 0, 0), (0, 0, look), (0, 1, 0), 40.0, W / H, 0.0, 1.0)
    return SceneArrays(cam, m, triangles=t)


def inside_sphere_scene(W, H):
    """The camera at the centre of a lambertian sphere of radius 10."""
    m = np.zeros(1, material_dtype)
    m[0]["albedo"] = (0.5, 0.5, 0.5)
    s = np.zeros(1, sphere_dtype)
    s[0] = ((0, 0, 0), 10.0, 0)
    return SceneArrays(camera_derive((0, 0, 0), (0, 0, -1), (0, 1, 0), 40.0, W / H, 0.0, 1.0), m, s)


def triangle_normal(tri):
    """orc_triangle_normal: the float unit face normal the product stores"""
    n = np.zeros(3, np.float32)
    t = np.ascontiguousarray(tri, dtype=triangle_dtype)
    oracle_lib().orc_triangle_normal(C.c_void_p(t.ctypes.data), C.c_void_p(n.ctypes.data))
    return n


def camera_dirs(orc, W, H, spp, seed, precision):
    """[spp, H*W, 3] float64: the oracle's camera-ray directions of every pixel and sample"""
    f = orc.camera_rays if precision == "f32" else orc.camera_rays_f64
    pix = np.arange(W * H)
    return np.stack([f(W, H, pix, s, seed)[:, 3:6].astype(np.float64) for s in range(spp)])


AOV_KEYS = ("albedo", "normal", "depth", "coverage")
_aov_lib = None


def aov_oracle_lib():
    """tests/aov_oracle.c, the AOV checker over the oracle's public entry points, built once per process into a temporary
    directory (the tree may be read-only) and linked against the oracle library the other tests load"""
    global _aov_lib
    if _aov_lib is None:
        oracle = os.path.abspath(build_oracle())
        oracle_lib()  # loaded first, so that the checker binds to the same copy
        so = os.path.join(tempfile.mkdtemp(prefix="aov_oracle_"), "libaov_oracle.so")
        subprocess.check_call(["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-I", ORACLE_DIR, os.path.join(ROOT, "tests", "aov_oracle.c"), "-o", so, oracle,
                               "-Wl,-rpath," + os.path.dirname(oracle), "-lm"])
        _aov_lib = C.CDLL(so)
    return _aov_lib


def oracle_aov(orc, W, H, spp, seed, use_bvh=True, rank=0, world=1, precision="f32"):
    """The first-hit AOVs of the CPU checker for the scene of Oracle `orc`: dict of float32 albedo [H, W, 3],
    normal [H, W, 3], depth [H, W], coverage [H, W], as Context.render_aov"""
    lib = aov_oracle_lib()
    out = dict(albedo=np.zeros((H, W, 3), np.float32), normal=np.zeros((H, W, 3), np.float32),
               depth=np.zeros((H, W), np.float32), coverage=np.zeros((H, W), np.float32))
    fn = lib.aov_render if precision == "f32" else lib.aov_d_render
    fn(C.byref(orc._s), orc.bvh() if use_bvh else None, W, H, spp, C.c_uint64(seed), rank, world,
       *[C.c_void_p(out[k].ctypes.data) for k in AOV_KEYS])
    return out


def aov_bytes(aov):
    return b"".join(np.ascontiguousarray(aov[k], np.float32).tobytes() for k in AOV_KEYS)


# ---------------------------------------------------------------------------------------------------------------
# anchors
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("use_bvh", [True, False])
def test_plane_anchor(precision, use_bvh):
    W, H, spp, seed = 16, 12, 4, 11
    sc = plane_scene(W, H)
    orc = Oracle(sc)
    aov = oracle_aov(orc, W, H, spp, seed, use_bvh=use_bvh, precision=precision)
    assert np.all(aov["coverage"] == 1.0)
    assert np.all(aov["albedo"] == np.array([0.2, 0.4, 0.6], np.float32))
    n = triangle_normal(sc.triangles[0])
    assert n[2] > 0.999 and np.array_equal(n, triangle_normal(sc.triangles[1]))  # (0, 0, +-1): towards the camera
    assert np.all(aov["normal"] == n)
    d = camera_dirs(orc, W, H, spp, seed, precision)
    want = (D * np.linalg.norm(d, axis=2) / np.abs(d[:, :, 2])).mean(axis=0).reshape(H, W)
    assert np.allclose(aov["depth"], want, rtol=1e-5, atol=0)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_all_miss_anchor(precision):
    W, H = 16, 12
    aov = oracle_aov(Oracle(plane_scene(W, H, look=1.0)), W, H, 3, 5, precision=precision)
    for k in AOV_KEYS:
        assert not np.any(aov[k]), k


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("mtype, albedo, want", [
    (LAMBERTIAN, (1.7, 1.7, 1.7), (1.0, 1.0, 1.0)),
    (LAMBERTIAN, (1.7, -0.5, 0.25), (1.0, 0.0, 0.25)),
    (DIFFUSE_LIGHT, (5.0, 5.0, 5.0), (1.0, 1.0, 1.0)),
    (DIELECTRIC, (0.1, 0.2, 0.3), (1.0, 1.0, 1.0)),
], ids=["albedo-1.7", "per-channel", "emitter-le5", "dielectric"])
def test_albedo_clamp_anchor(precision, mtype, albedo, want):
    W, H = 16, 12
    aov = oracle_aov(Oracle(plane_scene(W, H, mtype, albedo)), W, H, 3, 5, precision=precision)
    assert np.all(aov["albedo"] == np.array(want, np.float32))
    assert np.all(aov["coverage"] == 1.0)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_back_face_normals_point_at_the_camera(precision):
    """From inside a sphere every hit is a back face: the face-forwarded normal points inward, against the ray."""
    W, H, seed = 16, 12, 3
    orc = Oracle(inside_sphere_scene(W, H))
    aov = oracle_aov(orc, W, H, 1, seed, precision=precision)
    d = camera_dirs(orc, W, H, 1, seed, precision)[0]
    u = (d / np.linalg.norm(d, axis=1, keepdims=True)).reshape(H, W, 3)
    assert np.allclose(aov["normal"], -u, atol=1e-5)
    assert np.allclose(aov["depth"], 10.0, rtol=1e-5)


# ---------------------------------------------------------------------------------------------------------------
# consistency of the oracle: tree and scan, tile shards
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["final", "test3"])
def test_tree_and_scan_and_shards_agree(name, precision):
    W, H, spp, seed = 37, 21, 3, 9
    orc = Oracle(load_golden(name)[0])
    whole = oracle_aov(orc, W, H, spp, seed, use_bvh=True, precision=precision)
    assert aov_bytes(oracle_aov(orc, W, H, spp, seed, use_bvh=False, precision=precision)) == aov_bytes(whole)
    assert whole["coverage"].min() < 1.0 < 2 * whole["coverage"].max()  # some pixels see the sky, some geometry
    tile = (np.arange(H)[:, None] // 4) * ((W + 7) // 8) + np.arange(W)[None, :] // 8
    for world in (2, 3):
        total = {k: np.zeros_like(whole[k]) for k in AOV_KEYS}
        for rank in range(world):
            part = oracle_aov(orc, W, H, spp, seed, rank=rank, world=world, precision=precision)
            for k in AOV_KEYS:
                mine = tile % world == rank
                assert not np.any(part[k][~mine]), (world, rank, k)  # disjoint: other ranks' pixels stay 0
                total[k] += part[k]
        assert aov_bytes(total) == aov_bytes(whole), world


# ---------------------------------------------------------------------------------------------------------------
# pinned outputs (as tests/test_lights.py pins the framebuffers)
# ---------------------------------------------------------------------------------------------------------------
PIN_W, PIN_H, PIN_SPP, PIN_SEED = 24, 16, 3, 7
AOV_PINS = {
    "test2": {"f32": "af61fe99e6f7c418b69127db8c68fc6c873d3b6acf55b19588396a532442f013",
              "f64": "76fa93790cff93bf7d1344253abbbc4fce82b8729ea11c174f29a958deef4843"},
    "test3": {"f32": "67f6bbb6b4fa66f96a8638e784cfa75108d57e87af688c824fb889155b958e50",
              "f64": "eaf1302f2dbc5e5e59f440228dd206b46af2203b57d743707543b4c286701c8e"},
    "final": {"f32": "21f4447763e3aa29a10c4e0fa197e5fd70b59579faedc392682501ddc1fc96ba",
              "f64": "3d01dc6f47a9550dde8532c789ad0e05455651654682acd0e42deb5a6dc6e5df"},
    "cornell": {"f32": "7d99a8703228818d0a93b8e8b0973c0e9a124183c73ce3b8b7711a7a7e41833b",
                "f64": "8fd6a9572cc31dc49919319ef3d30f50120e27f056c5739547676c5d340c78c7"},
}


def pin_scene(name):
    if name == "cornell":
        from rrt_b200 import Scene

        return Scene.from_file(CORNELL, PIN_W, PIN_H).arrays
    return load_golden(name)[0]


def aov_digests(orc):
    return {p: hashlib.sha256(aov_bytes(oracle_aov(orc, PIN_W, PIN_H, PIN_SPP, PIN_SEED, precision=p))).hexdigest()
            for p in PRECISIONS}


@pytest.mark.parametrize("name", list(AOV_PINS))
def test_oracle_aov_outputs_are_pinned(name, request):
    """The oracle's four buffers of both integrators, at 24x16 and 3 spp, equal the digests computed when the AOVs were
    added.  The GPU is held to the oracle bit for bit, so only a change of the definition may change this table, in the
    same change as the kernel."""
    if name == "cornell":
        request.getfixturevalue("built_lib")
    assert aov_digests(Oracle(pin_scene(name))) == AOV_PINS[name]


# ---------------------------------------------------------------------------------------------------------------
# PFM writer, CLI
# ---------------------------------------------------------------------------------------------------------------
def read_pfm(path):
    """A minimal PFM reader: (header lines, float32 array [H, W, C] or [H, W] in file row order)"""
    raw = open(path, "rb").read()
    lines, pos = [], 0
    for _ in range(3):
        end = raw.index(b"\n", pos)
        lines.append(raw[pos:end].decode())
        pos = end + 1
    W, H = map(int, lines[1].split())
    ch = 3 if lines[0] == "PF" else 1
    scale = float(lines[2])
    a = np.frombuffer(raw[pos:], dtype="<f4" if scale < 0 else ">f4")
    assert a.size == W * H * ch
    return lines, a.reshape((H, W, ch) if ch == 3 else (H, W)).astype(np.float32), raw[pos:]


def test_pfm_round_trip(tmp_path, built_lib):
    from rrt_b200 import RrtbError, write_pfm

    rng = np.random.default_rng(1)
    rgb = rng.normal(size=(5, 7, 3)).astype(np.float32)
    rgb[0, 0] = [np.inf, -0.0, 1e-40]
    write_pfm(tmp_path / "c.pfm", rgb)
    lines, back, body = read_pfm(tmp_path / "c.pfm")
    assert lines == ["PF", "7 5", "-1.0"]
    assert body == rgb.astype("<f4").tobytes()  # rows bottom-up: the array's own row order, no flip
    assert back.tobytes() == rgb.tobytes()
    gray = rng.uniform(size=(3, 4)).astype(np.float32)
    write_pfm(tmp_path / "g.pfm", gray)
    lines, back, body = read_pfm(tmp_path / "g.pfm")
    assert lines == ["Pf", "4 3", "-1.0"] and body == gray.astype("<f4").tobytes()
    with pytest.raises(RrtbError):
        write_pfm(tmp_path / "no" / "such" / "dir.pfm", gray)
    from rrt_b200 import _lib

    lib = _lib.load()
    assert lib.rrtb_write_pfm(str(tmp_path / "x.pfm").encode(), 4, 3, 2, C.c_void_p(gray.ctypes.data)) == -1  # channels
    assert lib.rrtb_write_pfm(str(tmp_path / "x.pfm").encode(), 4, 3, 1, None) == -1


def test_cli_aov_usage_errors(built_lib):
    """-A without a value and -A with -I are usage errors (exit 1) found before any device is touched: without a GPU,
    touching one would exit 99."""
    if not os.path.exists(EXE):
        pytest.skip("drop-in executable not built")
    r = subprocess.run([EXE, "-A"], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage: rrt [options]" in r.stderr and "-A <prefix>" in r.stderr
    r = subprocess.run([EXE, "-A", "x", "-I", "list.txt"], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage: rrt [options]" in r.stderr
