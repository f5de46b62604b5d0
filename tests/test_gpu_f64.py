"""GPU parity tests of the DOUBLE integrator (SURVEY 8f1; RRTB_PRECISION_F64, what the reference's `rrtd` build
computes), through the C ABI, against oracle/rrt_oracle_f64.c -- itself pinned to the reference's double build in
tests/test_f64_oracle.py.

Bar: BIT-EXACT.  Every double operation on the device is an explicit round-to-nearest intrinsic in the oracle's
order, and IEEE add / mul / fma / div / sqrt are correctly rounded on both sides, so primary rays, closest hits,
hit records, scatter directions and whole framebuffers must be equal bit for bit.  Images additionally meet the
PSNR >= 40 dB bar against the reference's committed rrto renders.
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLD, ROOT, load_golden
from oracle_lib import Oracle, pinhole_rays, psnr

pytestmark = pytest.mark.gpu


def test_f64_camera_rays_bit_exact(ctx, golden):
    name, scene, d = golden
    W, H = int(d["W"]), int(d["H"])
    ctx.set_scene(scene)
    rng = np.random.default_rng(11)
    pix = rng.integers(0, W * H, size=1500).astype(np.int32)
    pix[:4] = [0, W - 1, W * (H - 1), W * H - 1]
    orc = Oracle(scene)
    for sample in (0, 7, 499):
        got = ctx.camera_rays_f64(W, H, pix, sample, seed=1984)
        want = orc.camera_rays_f64(W, H, pix, sample, 1984)
        assert got.tobytes() == want.tobytes(), (name, sample)


@pytest.mark.parametrize("mode", ["scan", "bvh"])
def test_f64_hits_bit_exact(ctx, golden, mode):
    """Primary rays of the configured image plus diffuse secondary rays leaving the first hits."""
    name, scene, d = golden
    W, H = int(d["W"]), int(d["H"])
    ctx.set_scene(scene, use_bvh=True)
    orc = Oracle(scene)
    rays = pinhole_rays(scene, W, H, step=5).astype(np.float64)
    if scene.camera["time0"][0] != scene.camera["time1"][0]:
        rays[:, 6] = np.random.default_rng(1).uniform(scene.camera["time0"][0], scene.camera["time1"][0], len(rays))
    for rnd in range(2):
        ids, t, rec = ctx.trace_f64(rays, 0.001, mode, want_rec=True)
        oid, ot, orec = orc.trace_f64(rays, 0.001, mode, want_rec=True)
        assert np.array_equal(ids, oid), (name, mode, rnd, int((ids != oid).sum()))
        assert t.tobytes() == ot.tobytes(), (name, mode, rnd)
        assert rec.tobytes() == orec.tobytes(), (name, mode, rnd)
        # next round: rays leaving the hit points (normal + random offset), like a lambertian bounce
        m = ids >= 0
        rng = np.random.default_rng(3)
        nxt = rays[m].copy()
        nxt[:, 0:3] = rec[m, 0:3]
        nxt[:, 3:6] = rec[m, 3:6] + 0.9 * rng.uniform(-1, 1, size=(m.sum(), 3)) / np.sqrt(3)
        rays = nxt


def test_f64_scatter_bit_exact(ctx, golden):
    name, scene, d = golden
    ctx.set_scene(scene)
    rng = np.random.default_rng(5)
    n = 4000
    nm = len(scene.materials)
    d_in = rng.normal(size=(n, 3)) * rng.uniform(0.2, 8, size=(n, 1))
    nrm = rng.normal(size=(n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    nrm[np.sum(d_in * nrm, axis=1) > 0] *= -1
    in16 = np.zeros((n, 16))
    in16[:, 0:3] = rng.uniform(-3, 3, size=(n, 3))
    in16[:, 3:6] = d_in
    in16[:, 7:10] = rng.uniform(-3, 3, size=(n, 3))
    in16[:, 10:13] = nrm
    in16[:, 13] = rng.integers(0, 2, size=n)
    in16[:, 14] = rng.integers(0, nm, size=n)
    rnd = rng.integers(0, 2**32, size=(n, 4), dtype=np.uint64).astype(np.uint32)
    got = ctx.scatter_f64(in16, rnd)
    want = Oracle(scene).scatter_f64(in16, rnd)
    assert got.tobytes() == want.tobytes(), name
    if name == "final":  # the scatter step's parameter space and edges (tests/test_scatter_space.py), once
        from test_scatter_space import cancel_inputs, space_inputs, space_scene

        space = space_scene()
        ctx.set_scene(space)
        orc = Oracle(space)
        in16, rnd, _ = space_inputs()
        c16, crnd = cancel_inputs(orc, "f64")
        for a, r in ((in16, rnd), (c16, crnd)):
            assert ctx.scatter_f64(a, r).tobytes() == orc.scatter_f64(a, r).tobytes()


def test_f64_render_bit_exact_vs_oracle(ctx, golden):
    """The whole estimator: camera -> traversal -> hit record -> scatter -> sky -> fixed-point sum, 50 bounces deep.
    The double framebuffer is accumulator * 2^-40 on both sides, so equality here is equality of every path."""
    name, scene, d = golden
    W, H, spp = 96, 64, 6
    orc = Oracle(scene)
    want, fixed, cnt = orc.render_f64(W, H, spp, 50, 1984)
    # LBVH with the state-machine kernel (default) and the one-segment-per-round kernel, then the flat scan
    for use_bvh, sched in ((True, 0), (True, 1), (False, 0)):
        ctx.set_scene(scene, use_bvh=use_bvh)
        for count in (True, False):
            img, st = ctx.render(W, H, spp, 50, seed=1984, count_rays=count, dtype=np.float64, precision="f64", scheduler=sched)
            assert st["paths"] == W * H * spp == cnt["paths"]
            if count:
                assert st["rays"] == cnt["rays"] and st["hits"] == cnt["hits"], (name, use_bvh, sched, st, cnt)
            assert img.tobytes() == want.tobytes(), (name, use_bvh, sched, count, float(np.abs(img - want).max()))
    # shallow depth cut-offs (rrt.cu:78) too
    ctx.set_scene(scene, use_bvh=True)
    for depth in (1, 3):
        img, _ = ctx.render(W, H, 2, depth, seed=7, dtype=np.float64, precision="f64")
        want, _, _ = orc.render_f64(W, H, 2, depth, 7)
        assert img.tobytes() == want.tobytes(), (name, depth)


def test_f64_render_shardable(ctx, golden):
    """Tile and sample shards of the double integrator sum to the single-GPU image bit for bit."""
    name, scene, d = golden
    W, H, spp = 90, 50, 5
    ctx.set_scene(scene)
    whole, _ = ctx.render(W, H, spp, 50, seed=3, dtype=np.float64, precision="f64")
    for shard_mode in (0, 1):
        acc = np.zeros_like(whole)
        for rank in range(3):
            part, st = ctx.render(W, H, spp, 50, seed=3, rank=rank, world=3, shard_mode=shard_mode, dtype=np.float64, precision="f64")
            acc += part
        # sums of fixed-point values scaled by 2^-40 are exact in double at this spp
        assert acc.tobytes() == whole.tobytes(), (name, shard_mode)


def test_f64_close_to_f32(ctx, golden):
    """Same Philox streams: the two integrators produce the same image except where a rounding difference sends
    a path elsewhere."""
    name, scene, d = golden
    W, H, spp = 120, 80, 8
    ctx.set_scene(scene)
    a, _ = ctx.render(W, H, spp, 50, seed=1984)
    b, _ = ctx.render(W, H, spp, 50, seed=1984, dtype=np.float64, precision="f64")
    ga = np.sqrt(a.astype(np.float64) / spp).clip(0, 1)
    gb = np.sqrt(b / spp).clip(0, 1)
    close = np.abs(ga - gb).max(axis=2) < 1e-3
    assert close.mean() > 0.97, (name, close.mean())
    assert abs(ga.mean() - gb.mean()) < 2e-3


GOLDEN_RENDERS = {
    "test1": ("test1_480x320_s256_rrto.png", 480, 320, 256),
    "final": ("final_600x400_s500_rrto.png", 600, 400, 500),
}


@pytest.mark.parametrize("name", list(GOLDEN_RENDERS))
def test_f64_psnr_vs_reference_render(ctx, name):
    from PIL import Image

    from rrt_b200 import tonemap
    from test_gpu_parity import _scene_for

    fn, W, H, spp = GOLDEN_RENDERS[name]
    ref = np.asarray(Image.open(os.path.join(GOLD, fn)).convert("RGB"))
    ctx.set_scene(_scene_for(name, W, H), use_bvh=True)
    img, st = ctx.render(W, H, spp, 50, seed=1984, dtype=np.float64, precision="f64")
    ours = tonemap(img, spp)
    val = psnr(ours, ref)
    assert val >= 40.0, (name, val)
    assert abs(ours.astype(np.float64).mean() - ref.astype(np.float64).mean()) < 0.5


def test_f64_cli_rrtd(tmp_path, built_lib):
    """`rrtd` = the double integrator + double framebuffer + double tonemap, same pixels as the API."""
    from PIL import Image

    from oracle_lib import ref_scene_path
    from rrt_b200 import Context, Scene, tonemap

    exe = os.path.join(ROOT, "rrt_b200", "bin", "rrtd")
    scene_path = ref_scene_path("test2.txt")
    if not (os.path.exists(exe) and scene_path):
        pytest.skip("drop-in executable or scene text not staged")
    out = tmp_path / "t.png"
    r = subprocess.run([exe, "-i", scene_path, "-o", str(out), "-w", "96", "-h", "54", "-s", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert ",double," in r.stderr
    png = np.asarray(Image.open(out).convert("RGB"))
    with Context(0) as c:
        c.set_scene(Scene.from_file(scene_path, 96, 54))
        img, _ = c.render(96, 54, 3, 50, seed=1984, dtype=np.float64, precision="f64")
    assert np.array_equal(png, tonemap(img, 3))
