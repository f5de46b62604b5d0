"""The float integrator held to the double one path by path (CPU: the float oracle against the double oracle).

Both integrators draw the same Philox streams, so at 1 spp the float path and the double path of a pixel hit the same
sequence of surfaces, except where rounding flips a discrete decision: a silhouette, the critical angle, the Schlick
draw, the absorption sign.  A render with a double framebuffer returns each one-path pixel as its exact 2^-40
fixed-point value, so the two renders compare path by path:

    rel = max(max_c |a - b| - 2^-39, 0) / max_c |b|      (two fixed-point quanta forgiven: deep, dim paths)

A path diverges when rel > 1e-3 or when exactly one of the two is black.  Bars: at depth 1 every path agrees to 1e-6
(the sky through a float reciprocal square root) and the escape sets differ by at most 1e-5 of the paths (camera rays
grazing a silhouette: 1 of 153 600 on final.txt); at depths 2 and 50 at most 0.2 % of the paths diverge, the 99.9th
percentile of rel over the agreeing paths is <= 3e-4, and the mean relative difference of the channel sums over the
agreeing paths is <= 1e-6 -- a one-sided rounding (a throughput narrowed to 16 bits, a scaled sky) that a two-sided
1e-3 bar lets through.  tests/test_gpu_path_by_path.py holds the GPU's float integrator to the same statistic, with the
float oracle's numbers on the same case, computed here, as its yardstick.
"""
import functools
import os
import tempfile

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle_lib import Oracle
from rrt_b200.types import SceneArrays

W, H = 480, 320
SEEDS = (1984, 2**32 + 1984)
DEPTHS = (1, 2, 50)
NAMES = ("final", "test2", "test3", "fast", "mtri", "cornell", "gain", "varied")
FLOOR = 2.0**-39  # two quanta of the 2^40 fixed point
DIVERGE = 1e-3
DEPTH1_REL = 1e-6
P999_REL = 3e-4  # the float oracle: 1.6e-4 .. 1.9e-4 on final.txt and its variants at depth 50, <= 7e-6 elsewhere
BIAS = 1e-6
ORACLE_DIVERGED = 2e-3
ESCAPE_MISMATCH = 1e-5  # depth 1: camera rays that graze a silhouette can hit in one precision and miss in the other

VARIED_FUZZ = (-0.7, 0.0, 0.3, 1.0, 1.8)
VARIED_IR = (1 / 1.5, 1.0, 1.33, 2.42)


def varied_scene():
    """final.txt with its metals' fuzz drawn from VARIED_FUZZ and its glass indices from VARIED_IR (every value
    occurs; fixed rng)."""
    sc, _ = load_golden("final")
    m = sc.materials.copy()
    rng = np.random.default_rng(2024)
    metal, glass = np.nonzero(m["type"] == 1)[0], np.nonzero(m["type"] == 2)[0]
    m["param"][metal] = rng.permutation(np.resize(VARIED_FUZZ, len(metal)))
    m["param"][glass] = rng.permutation(np.resize(VARIED_IR, len(glass)))
    return SceneArrays(sc.camera, m, sc.spheres, sc.mspheres, sc.triangles, sc.mtriangles)


@functools.lru_cache(maxsize=None)
def path_scene(name):
    """The scenes of the per-path comparison: the three golden scenes, 64 fast spheres (motion nodes), 8 moving
    triangles (the MTRI kernels), cornell.txt (the LIGHTS kernels), final.txt at 3x albedo (samples that reach the
    clamp) and final.txt with varied fuzz and indices."""
    if name in ("final", "test2", "test3"):
        return load_golden(name)[0]
    if name == "varied":
        return varied_scene()
    if name == "fast":
        from test_moving_instances import fast_spheres_scene

        return fast_spheres_scene()
    if name == "gain":
        from test_gpu_launch_space import gain_scene

        return gain_scene()
    from rrt_b200 import Scene

    if name == "cornell":
        return Scene.from_file(os.path.join(ROOT, "scenes", "cornell.txt"), W, H).arrays
    assert name == "mtri"
    from test_moving_instances import scene_text

    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "mtri.txt")
        with open(p, "w") as f:
            f.write(scene_text("moving"))
        return Scene.from_file(p, W, H).arrays


@functools.lru_cache(maxsize=None)
def oracle_paths(name, seed, depth):
    """(float oracle, double oracle) one-path pixels [H, W, 3] as float64 values of their fixed-point sums."""
    orc = Oracle(path_scene(name))
    _, f32, c32 = orc.render(W, H, 1, depth, seed)
    _, f64, c64 = orc.render_f64(W, H, 1, depth, seed)
    assert c32["paths"] == c64["paths"] == W * H
    return f32.astype(np.float64) * 2.0**-40, f64.astype(np.float64) * 2.0**-40


def path_stats(a, b):
    """The float paths `a` against the double paths `b`: diverged fraction, 99.9th percentile of rel and the mean
    relative difference of the channel sums over the agreeing (non-black) paths, the paths black on one side only, and
    the worst rel over the others."""
    a, b = a.reshape(-1, 3), b.reshape(-1, 3)
    err = np.maximum(np.abs(a - b).max(axis=1) - FLOOR, 0.0)
    mb = np.abs(b).max(axis=1)
    rel = np.where(mb > 0, err / np.where(mb > 0, mb, 1.0), 0.0)
    black_a, black_b = ~(a > 0).any(axis=1), ~(b > 0).any(axis=1)
    one_black = black_a != black_b
    diverged = one_black | (rel > DIVERGE)
    agree = ~diverged
    lit = agree & ~black_b
    sa, sb = a.sum(axis=1), b.sum(axis=1)
    return dict(
        paths=len(a), diverged=float(diverged.mean()), diverged_1e2=float((one_black | (rel > 1e-2)).mean()),
        one_black=int(one_black.sum()), worst=float(rel[~one_black].max()),
        p999=float(np.quantile(rel[agree], 0.999)) if agree.any() else 0.0,
        bias=float(np.mean((sa[lit] - sb[lit]) / sb[lit])) if lit.any() else 0.0, lit=int(lit.sum()),
    )


def check_paths(s, depth, max_diverged, max_p999, label):
    print("%s: diverged %.5f %% (%.5f %% above 1e-2), p99.9 rel %.2e, bias %+.2e over %d lit paths, worst %.2e, "
          "%d black on one side" % (label, 100 * s["diverged"], 100 * s["diverged_1e2"], s["p999"], s["bias"], s["lit"],
                                    s["worst"], s["one_black"]))
    assert s["lit"] >= 500, (label, s)
    if depth == 1:  # the sky (or an emitter) of the same segment
        assert s["one_black"] <= ESCAPE_MISMATCH * s["paths"], (label, s)
        assert s["worst"] <= DEPTH1_REL, (label, s)
        return
    assert s["diverged"] <= max_diverged, (label, s, max_diverged)
    assert s["p999"] <= max_p999, (label, s, max_p999)
    assert abs(s["bias"]) <= BIAS, (label, s)


CASES = [(n, s, d) for n in NAMES for s in SEEDS for d in DEPTHS]


def case_id(c):
    return "%s-seed%d-d%d" % c


def test_varied_scene_has_every_value():
    m = varied_scene().materials
    assert set(m["param"][m["type"] == 1].tolist()) == set(np.float32(VARIED_FUZZ).tolist())
    assert set(m["param"][m["type"] == 2].tolist()) == set(np.float32(VARIED_IR).tolist())


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_float_oracle_path_by_path(case, built_lib):
    name, seed, depth = case
    a, b = oracle_paths(name, seed, depth)
    check_paths(path_stats(a, b), depth, ORACLE_DIVERGED, P999_REL, "float oracle " + case_id(case))
