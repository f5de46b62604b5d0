"""Writes tests/golden/scenes/{test1,test2,test3,final}.txt: stand-ins for the reference's four scene files, which the
repository does not ship.  Each is written from what the reference's own parser built from the original file
(tests/golden/scene_<name>.npz), and is checked to parse back, through the product's parser, to exactly those arrays
and object counts.  The texts are not the originals (fewer lines, other number spellings, test2's obj block holds the
already transformed vertices of its first instance); a scene parsed from them is the reference's scene bit for bit.

    python tools/make_scene_texts.py [out_dir]        (needs the built library: __graft_entry__.build())
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rrt_b200 import Scene  # noqa: E402
from rrt_b200.types import SceneArrays  # noqa: E402

# lookfrom, lookat, vup, vfov, aperture, focus [, time0 time1]: the camera lines whose derivation gives the stored
# camera records bit for bit
CAMERAS = {
    "test1": "0 2 5  0 0 -1  0 1 0  30 0.1 6",
    "test2": "-1 2 5  0 0.5 -1  0 1 0  30 0.1 6",
    "test3": "0 2 5  0 0 -1  0 1 0  30 0.1 6 0 0.5",
    "final": "13 2 3  0 0 0  0 1 0  30 0.1 10",
}
FIELDS = ("camera", "materials", "spheres", "mspheres", "triangles")
COUNTS = ("materials", "spheres", "mspheres", "triangles", "objs", "obj_insts")


def num(x):
    """The shortest decimal that names this float32 (read back through double, as the parser does)."""
    return np.format_float_positional(np.float32(x), unique=True, trim="-")


def nums(v):
    return " ".join(num(x) for x in v)


def scene_text(name, s: SceneArrays, obj_size=4):
    lines = ["camera " + CAMERAS[name]]
    for i, m in enumerate(s.materials):
        kind = int(m["type"])
        if kind == 0:
            lines.append("material m%d lambertian %s" % (i, nums(m["albedo"])))
        elif kind == 1:
            lines.append("material m%d metal %s %s" % (i, nums(m["albedo"]), num(m["param"])))
        else:
            lines.append("material m%d dielectric %s" % (i, num(m["param"])))
    for sp in s.spheres:
        lines.append("sphere %s %s m%d" % (nums(sp["center"]), num(sp["radius"]), sp["material"]))
    for ms in s.mspheres:
        lines.append("msphere %s %s %s %s %s m%d" % (nums(ms["center0"]), nums(ms["center1"]), num(ms["time0"]), num(ms["time1"]),
                                                    num(ms["radius"]), ms["material"]))
    t = s.triangles
    if len(t):  # test2: one obj of obj_size triangles, instanced by translation
        base = t[:obj_size]
        verts = []
        for tri in base:
            for k in ("v0", "v1", "v2"):
                if tuple(tri[k].tolist()) not in verts:
                    verts.append(tuple(tri[k].tolist()))
        lines.append("obj_beg %d %d" % (len(verts), len(base)))
        lines += ["obj_vtx " + nums(v) for v in verts]
        lines += ["obj_tri " + " ".join(str(verts.index(tuple(tri[k].tolist()))) for k in ("v0", "v1", "v2")) for tri in base]
        lines.append("obj_end")
        for g in range(0, len(t), obj_size):
            d = (t[g]["v0"] - t[0]["v0"]).astype(np.float64)
            lines.append("obj 0 m%d" % t[g]["material"] + ("" if not d.any() else " t " + nums(np.round(d, 4))))
    return "\n".join(lines) + "\n"


def main(out):
    os.makedirs(out, exist_ok=True)
    for name in CAMERAS:
        d = np.load(os.path.join(ROOT, "tests", "golden", "scene_%s.npz" % name))
        want = SceneArrays.from_npz_dict(d)
        path = os.path.join(out, name + ".txt")
        with open(path, "w") as f:
            f.write(scene_text(name, want))
        got = Scene.from_file(path, int(d["W"]), int(d["H"]))
        bad = [k for k in FIELDS if getattr(got.arrays, k).tobytes() != getattr(want, k).tobytes()]
        c = got.counts()
        if bad or [c[k] for k in COUNTS] != d["counts"].tolist():
            sys.exit("%s: %s does not parse back to the stored scene (%s)" % (name, path, bad or "counts"))
        print("%s: %s" % (name, path))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "scenes"))
