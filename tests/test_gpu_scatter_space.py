"""The GPU's scatter hooks across the scatter step's parameter space (-m gpu); inputs and checks are those of
tests/test_scatter_space.py.  The double hook equals the double oracle bit for bit on these inputs in
tests/test_gpu_f64.py::test_f64_scatter_bit_exact.

The float hook may use rsqrtf and __fdividef (each within 2 ulp): its direction budget against the double oracle is
the float oracle's K plus 4 ulp, and the worst ratio seen is printed.
"""
import numpy as np
import pytest

from oracle_lib import Oracle
from test_scatter_space import (DIST_CASES, K_GPU, anchors, cancel_inputs, check_cancel, check_distribution, compare,
                                dist_id, space_inputs, space_scene)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def space(ctx):
    scene = space_scene()
    ctx.set_scene(scene)
    in16, rnd, kind = space_inputs()
    return scene, Oracle(scene), in16, rnd, kind


def test_gpu_float_scatter_against_double_oracle(ctx, space):
    scene, orc, in16, rnd, kind = space
    ctx.set_scene(scene)
    lo = ctx.scatter(in16.astype(np.float32), rnd)
    hi = orc.scatter_f64(in16, rnd)
    worst, n, ratio, ok = compare(lo, hi, in16, rnd, scene.materials, "GPU float")
    ref, _, _, _ = compare(orc.scatter(in16.astype(np.float32), rnd), hi, in16, rnd, scene.materials, "float oracle")
    print("GPU float scatter vs double oracle: worst %.3f x 2^-24 (|d64| + 1 + 1/|k|) over %d rows (float oracle %.3f)"
          % (worst, n, ref))
    assert n > 0.98 * len(in16)
    assert worst <= K_GPU


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_gpu_anchors(ctx, space, precision):
    scene, orc, in16, rnd, kind = space
    ctx.set_scene(scene)
    out = ctx.scatter(in16.astype(np.float32), rnd) if precision == "f32" else ctx.scatter_f64(in16, rnd)
    anchors(out, in16, rnd, kind, scene.materials, 12 if precision == "f32" else 4, "GPU " + precision)
    c16, crnd = cancel_inputs(orc, precision)
    out = ctx.scatter(c16.astype(np.float32), crnd) if precision == "f32" else ctx.scatter_f64(c16, crnd)
    exact = check_cancel(out, c16, "GPU " + precision)
    print("GPU %s: %d of %d cancelling lambertian rows return exactly n (the rest a residual of n + u below 2^-24)"
          % (precision, exact, len(c16)))
    if precision == "f64":
        assert exact == len(c16)  # as the double oracle does


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("case", DIST_CASES, ids=dist_id)
def test_gpu_distributions(ctx, space, case, precision):
    scene = space[0]
    ctx.set_scene(scene)
    if precision == "f32":
        fn = lambda a, r: ctx.scatter(a.astype(np.float32), r)
    else:
        fn = ctx.scatter_f64
    check_distribution(case, fn, scene.materials, K_GPU, "GPU " + precision)
