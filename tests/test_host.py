"""-m "not gpu": the host side of the drop-in (C++ inside librrtb200.so): scene parser with the reference
grammar + quirks, camera derivation, tonemap, PNG writer, CLI exit codes."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLD, ROOT, load_golden
from oracle_lib import ref_scene_path

EXE = os.path.join(ROOT, "rrt_b200", "bin", "rrt")


@pytest.mark.parametrize("name", ["test1", "test2", "test3", "final"])
def test_parser_bit_exact_vs_reference_parse(name, built_lib):
    """The four shipped scenes parse to exactly the arrays the reference's own parser produced (fixture).  Where the
    reference's files are not staged (oracle/_ref/scenes), the stand-ins of tests/golden/scenes are parsed: texts
    written from that fixture by tools/make_scene_texts.py, so this checks the parser on them, not on the originals."""
    from rrt_b200 import Scene

    p = ref_scene_path(name + ".txt")
    if not p:
        pytest.skip("scene text not staged")
    gold, d = load_golden(name)
    s = Scene.from_file(p, int(d["W"]), int(d["H"]))
    for k in ("camera", "materials", "spheres", "mspheres", "triangles"):
        assert getattr(s.arrays, k).tobytes() == getattr(gold, k).tobytes(), (name, k)
    c = s.counts()
    assert [c[k] for k in ("materials", "spheres", "mspheres", "triangles", "objs", "obj_insts")] == d["counts"].tolist()


def _write(tmp_path, text):
    p = tmp_path / "s.txt"
    p.write_text(text)
    return str(p)


CAM = "camera 0 2 5  0 0 -1  0 1 0  30 0.1 6\n"
MAT = "material m lambertian 0.5 0.5 0.5\n"


def test_parser_error_codes(tmp_path, built_lib):
    """exit codes of the reference: 2 cannot open (scene.h:220-223), 3 unknown material type (287-290),
    4 no camera / materials / objects (431-442), 1 obj errors (80-106,346-349)."""
    from rrt_b200 import Scene, SceneError

    cases = [
        (None, 2),
        (CAM + "material m plastic 1 1 1\nsphere 0 0 0 1 m\n", 3),
        (MAT + "sphere 0 0 0 1 m\n", 4),
        (CAM + "sphere 0 0 0 1 m\n", 4),
        (CAM + MAT, 4),
        (CAM + MAT + "obj_beg 3 1\nobj_vtx 0 0 0\nobj_vtx 1 0 0\nobj_end\n", 1),
        (CAM + MAT + "obj_vtx 0 0 0\n", 1),
        (CAM + MAT + "obj_beg 3 1\nobj_beg 3 1\n", 1),
        (CAM + MAT + "obj_beg 1 0\nobj_vtx 0 0 0\nobj_vtx 0 0 0\n", 1),
    ]
    for text, code in cases:
        path = "/nonexistent/scene.txt" if text is None else _write(tmp_path, text)
        with pytest.raises(SceneError) as e:
            Scene.from_file(path, 120, 80)
        assert e.value.ref_exit_code == code, (text, e.value.ref_exit_code)


def test_parser_quirks(tmp_path, built_lib):
    """SURVEY Appendix A: prefix dispatch at column 0, last camera wins, unknown material name -> index 0,
    first definition of a duplicate material name wins, transforms applied in listed order, rotation about
    the axis as given, shutter times optional."""
    from rrt_b200 import Scene

    text = (
        "# comment\n"
        "   sphere 9 9 9 9 m\n"  # leading whitespace: ignored
        "camera 0 0 9  0 0 0  0 1 0  10 0 1\n" + CAM.replace("6\n", "6 0.25 0.75\n") +
        "material a lambertian 0.1 0.2 0.3\nmaterial b metal 0.4 0.5 0.6 2.5\nmaterial a dielectric 1.5\n"
        "sphere 1 2 3 4 b\nsphere 0 0 0 1 nosuch\nsphere 0 0 0 1 a\n"
        "msphere 0 0 0  1 1 1  0.5 1.5  0.25 b\n"
        "obj_beg 3 1\nobj_vtx 1 0 0\nobj_vtx 0 1 0\nobj_vtx 0 0 1\nobj_tri 0 1 2\nobj_end\n"
        "obj 0 b s 2 2 2 t 1 0 0\nobj 0 a t 1 0 0 s 2 2 2\nobj 0 a r 90 0 0 1\n"
    )
    s = Scene.from_file(_write(tmp_path, text), 300, 200)
    a = s.arrays
    assert len(a.spheres) == 3 and len(a.materials) == 3 and len(a.mspheres) == 1 and len(a.triangles) == 3
    assert a.spheres["material"].tolist() == [1, 0, 0]  # 'nosuch' -> 0; 'a' -> first definition (index 0)
    assert a.materials["type"].tolist() == [0, 1, 2] and a.materials["param"][1] == np.float32(2.5)
    assert (a.camera["time0"][0], a.camera["time1"][0]) == (np.float32(0.25), np.float32(0.75))
    assert np.allclose(a.camera["origin"][0], (0, 2, 5))  # last camera line wins
    assert np.allclose(a.triangles["v0"][0], (3, 0, 0)) and np.allclose(a.triangles["v0"][1], (4, 0, 0))
    assert np.allclose(a.triangles["v0"][2], (0, 1, 0), atol=1e-6)  # (1,0,0) rotated 90 deg about z
    assert s.counts()["objs"] == 1 and s.counts()["obj_insts"] == 3
    assert a.mspheres["time1"][0] == np.float32(1.5) and a.mspheres["radius"][0] == np.float32(0.25)


def test_tonemap_and_png_roundtrip(tmp_path, built_lib):
    from PIL import Image

    from rrt_b200 import tonemap, write_png

    k = np.load(os.path.join(GOLD, "kat_math.npz"))
    sums = k["tm_sums"]
    img = tonemap(sums.reshape(1, -1, 3), int(k["tm_spp"]))
    assert np.array_equal(img.reshape(-1, 3).astype(np.int32), k["tm_rgb"])  # == reference convert_color
    rng = np.random.default_rng(0)
    fb = rng.uniform(0, 8, size=(37, 53, 3)).astype(np.float32)
    rgb = tonemap(fb, 8)
    ref = (256 * np.clip(np.sqrt(fb / np.float32(8)), 0, 0.999)).astype(np.uint8)[::-1]  # flip: row 0 = bottom
    assert np.abs(rgb.astype(int) - ref.astype(int)).max() <= 1
    p = tmp_path / "x.png"
    write_png(p, rgb)
    assert np.array_equal(np.asarray(Image.open(p).convert("RGB")), rgb)


def test_cli_exit_codes(tmp_path, built_lib):
    """usage + exit 1 on unknown flags / missing scene (main.cpp:33-51,126-127); parser codes pass through."""
    if not os.path.exists(EXE):
        pytest.skip("drop-in executable not built")
    r = subprocess.run([EXE, "-z"], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage: rrt [options]" in r.stderr and "Unexpected argument: -z" in r.stderr
    r = subprocess.run([EXE], capture_output=True, text=True)
    assert r.returncode == 1 and "ERROR: no scene loaded." in r.stderr
    r = subprocess.run([EXE, "stray"], capture_output=True, text=True)
    assert r.returncode == 1
    r = subprocess.run([EXE, "-i", "/nonexistent.txt"], capture_output=True, text=True)
    assert r.returncode == 2 and "ERROR: problem with opening file" in r.stderr
    r = subprocess.run([EXE, "-i", _write(tmp_path, CAM + "material m plastic 1\n")], capture_output=True, text=True)
    assert r.returncode == 3
    r = subprocess.run([EXE, "-i", _write(tmp_path, CAM + MAT)], capture_output=True, text=True)
    assert r.returncode == 4
    import torch

    if not torch.cuda.is_available():
        # valid scene, no GPU: the renderer must fail loudly with the reference's CUDA-failure code (rrt.cu:39)
        p = ref_scene_path("test1.txt")
        if p:
            r = subprocess.run([EXE, "-i", p, "-w", "32", "-h", "16", "-s", "1", "-input-alias-check"], capture_output=True, text=True)
            assert r.returncode in (1, 99)
            r = subprocess.run([EXE, "-input", p, "-w", "32", "-h", "16", "-s", "1"], capture_output=True, text=True)
            assert r.returncode == 99 and "no CPU fallback" in r.stderr and "sphere count:    4" in r.stderr


# ---------------------------------------------------------------------------------------------------------------
# parser fuzz against the LIVE reference parser (oracle/_ref/libref_f.so = scene.h compiled as is)
# ---------------------------------------------------------------------------------------------------------------
def _num(rng, lo, hi):
    """One number in one of the spellings std::stod accepts."""
    v = rng.uniform(lo, hi)
    style = rng.integers(0, 6)
    if style == 0:
        return "%d" % round(v)
    if style == 1:
        return "%.3f" % v
    if style == 2:
        return "%.6e" % v
    if style == 3:
        return ("+" if v >= 0 else "") + "%.2f" % v
    if style == 4:
        return repr(float(np.float32(v)))
    return "%.10f" % v


def _random_scene_text(seed):
    rng = np.random.default_rng(seed)
    sep = lambda: " " * int(rng.integers(1, 4)) if rng.uniform() < 0.8 else "\t"
    L = []
    join = lambda *w: sep().join(str(x) for x in w) + (" " * int(rng.integers(0, 3)))
    L.append("# fuzz scene %d" % seed)
    times = [_num(rng, 0, 0.4), _num(rng, 0.5, 1.5)] if rng.uniform() < 0.5 else []
    L.append(join("camera", *[_num(rng, -6, 6) for _ in range(3)], *[_num(rng, -1, 1) for _ in range(3)], 0, 1, 0, _num(rng, 15, 60),
                  _num(rng, 0, 0.3), _num(rng, 2, 9), *times))
    names = []
    for k in range(int(rng.integers(1, 7))):
        n = "m%d" % k
        kind = rng.integers(0, 3)
        if kind == 0:
            L.append(join("material", n, "lambertian", *[_num(rng, 0, 1) for _ in range(3)]))
        elif kind == 1:
            L.append(join("material", n, "metal", *[_num(rng, 0, 1) for _ in range(3)], _num(rng, 0, 1.5)))
        else:
            L.append(join("material", n, "dielectric", _num(rng, 1.1, 2.4)))
        names.append(n)
        if rng.uniform() < 0.3:
            L.append("")
        if rng.uniform() < 0.2:
            L.append("   sphere 0 0 0 1 %s" % n)  # leading blank: the line is ignored (prefix must sit at column 0)
    pick = lambda: names[int(rng.integers(0, len(names)))]
    n_obj = int(rng.integers(0, 3))
    for o in range(n_obj):
        nv, nt = int(rng.integers(3, 7)), int(rng.integers(1, 6))
        L.append(join("obj_beg", nv, nt))
        for _ in range(nv):
            L.append(join("obj_vtx", *[_num(rng, -1, 1) for _ in range(3)]))
        for _ in range(nt):
            L.append(join("obj_tri", *[int(x) for x in rng.choice(nv, 3, replace=False)]))
        L.append("obj_end")
    for _ in range(int(rng.integers(1, 9))):
        L.append(join("sphere", *[_num(rng, -5, 5) for _ in range(3)], _num(rng, 0.1, 2), pick()))
    for _ in range(int(rng.integers(0, 4))):
        L.append(join("msphere", *[_num(rng, -5, 5) for _ in range(6)], _num(rng, 0, 0.5), _num(rng, 0.6, 2), _num(rng, 0.1, 1), pick()))
    for _ in range(int(rng.integers(0, 5)) if n_obj else 0):
        xf = []
        for _ in range(int(rng.integers(0, 4))):
            op = "tsr"[int(rng.integers(0, 3))]
            if op == "r":
                xf += ["r", _num(rng, -180, 180), *[_num(rng, -1, 1) for _ in range(3)]]
            elif op == "s":
                xf += ["s", *[_num(rng, 0.2, 3) for _ in range(3)]]
            else:
                xf += ["t", *[_num(rng, -4, 4) for _ in range(3)]]
        L.append(join("obj", int(rng.integers(0, n_obj)), pick(), *xf))
    L.append("# end")
    return "\n".join(L) + "\n"


@pytest.mark.parametrize("seed", range(25))
def test_parser_fuzz_vs_live_reference_parser(seed, tmp_path, built_lib):
    """Random valid scene files (every number spelling std::stod takes, ragged whitespace, comments, ignored lines,
    obj blocks with translate / scale / rotate chains): camera, materials and every primitive bit-identical to what
    the reference's own parser (scene.h, compiled unmodified) builds."""
    from oracle_lib import RefScene, have_ref
    from rrt_b200 import Scene

    if not have_ref():
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    W, H = [(640, 360), (1200, 800), (333, 217)][seed % 3]
    path = _write(tmp_path, _random_scene_text(1000 + seed))
    ref = RefScene(path, W, H, "f")
    want = ref.arrays()
    got = Scene.from_file(path, W, H)
    for k in ("camera", "materials", "spheres", "mspheres", "triangles"):
        assert getattr(got.arrays, k).tobytes() == getattr(want, k).tobytes(), (seed, k)
    c = got.counts()
    assert [c[k] for k in ("materials", "spheres", "mspheres", "triangles", "objs", "obj_insts")] == [ref.counts[k] for k in ("materials", "spheres", "mspheres", "triangles", "objs", "obj_insts")]


def test_parser_survives_mutated_scenes_under_sanitizers():
    """tools/fuzz_parser.sh: rrtb_host.cpp built with AddressSanitizer + UBSan parses 300 mutated copies of the reference's
    scenes (truncated, shuffled, keyword / nan / inf / huge-number substitutions, random bytes): it may reject them, it
    may not crash, read out of bounds or leak."""
    import shutil

    scenes = os.path.dirname(ref_scene_path("final.txt"))
    if shutil.which("g++") is None:
        pytest.skip("needs g++")
    r = subprocess.run(["bash", os.path.join(ROOT, "tools", "fuzz_parser.sh"), "300", scenes], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "sanitizer findings 0" in r.stdout
