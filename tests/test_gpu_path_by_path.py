"""The GPU's float integrator held to its double integrator path by path (-m gpu); the statistic and the scenes are
those of tests/test_path_by_path.py.

Each case renders 480x320 at 1 spp with the float integrator through the pool kernel (the other schedulers give the
same bits: test_gpu_launch_space.py) and with the double integrator, both into the double framebuffer, so every pixel
is one path's exact fixed-point value.  The double render must equal the double oracle's bit for bit.  Bars against
the float oracle on the same scene, seed and depth:
  * depth 1: the GPU's escape set is the float oracle's (same camera rays, same hits), every other path within 1e-6;
  * depths 2 and 50: diverged fraction <= max(3 x the float oracle's, 1e-4); 99.9th percentile of rel over the agreeing
    paths <= max(1e-4, 2 x the float oracle's); mean relative difference of the channel sums <= 1e-6.
"""
import numpy as np
import pytest

from test_path_by_path import CASES, W, H, case_id, check_paths, oracle_paths, path_scene, path_stats

pytestmark = pytest.mark.gpu

POOL = 2  # RRTB_SCHED_POOL


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_gpu_float_integrator_path_by_path(ctx, case):
    name, seed, depth = case
    ctx.set_scene(path_scene(name), use_bvh=True)
    a, _ = ctx.render(W, H, 1, depth, seed=seed, scheduler=POOL, dtype=np.float64, precision="f32")
    b, _ = ctx.render(W, H, 1, depth, seed=seed, scheduler=POOL, dtype=np.float64, precision="f64")
    o32, o64 = oracle_paths(name, seed, depth)
    assert b.tobytes() == o64.tobytes(), case  # the double integrator is the double oracle
    ref = path_stats(o32, o64)
    s = path_stats(a, b)
    print("float oracle %s: diverged %.5f %%, p99.9 rel %.2e, bias %+.2e" % (case_id(case), 100 * ref["diverged"], ref["p999"], ref["bias"]))
    check_paths(s, depth, max(3 * ref["diverged"], 1e-4), max(1e-4, 2 * ref["p999"]), "GPU " + case_id(case))
    if depth == 1:
        assert np.array_equal((a > 0).any(axis=2), (o32 > 0).any(axis=2)), case
