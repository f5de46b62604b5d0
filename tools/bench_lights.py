#!/usr/bin/env python
"""Throughput of scenes with lights (the LIGHTS render kernels), one GPU.

    python tools/bench_lights.py [--steps K] [--warmup W] [--out FILE.jsonl]

Workloads, each in the float and the double integrator:
  cornell       scenes/cornell.txt (walls and a ceiling light, background 0 0 0), 800x800, 64 spp, depth 50
  final         final.txt 1200x800, 100 spp, depth 50: the sky kernels
  final+buried  the same scene plus `material l diffuse_light 5 5 5` and a sphere of radius 1 at (0, -900, 0), inside
                the ground sphere where no path reaches it: the same image through the LIGHTS kernel, so the ratio of the
                two rows is the LIGHTS kernel's overhead on a scene without visible lights
Rays come from one counting render; the time is the median device time (CUDA events) of K renders without counting.
final and final+buried alternate step by step.  The device name and power limit are read in the same run and printed
with every row.  Writes nothing unless --out is given.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import load_workload  # noqa: E402
from rrt_b200 import Context, Scene  # noqa: E402
from rrt_b200.types import DIFFUSE_LIGHT, SceneArrays, material_dtype, sphere_dtype  # noqa: E402


def buried_light(sc):
    m = np.concatenate([sc.materials, np.array([(DIFFUSE_LIGHT, (5, 5, 5), 0)], material_dtype)])
    s = np.concatenate([sc.spheres, np.array([((0, -900, 0), 1.0, len(m) - 1)], sphere_dtype)])
    return SceneArrays(sc.camera, m, s, sc.mspheres, sc.triangles, sc.mtriangles)


def device_facts(ctx):
    name = ctx.device_info()["name"]
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60).stdout.strip().split(",")
        return name, float(q[0]), float(q[1])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return name, None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    ctxs = {}
    final, _ = load_workload("final", 1200, 800)
    scenes = {
        "cornell": (Scene.from_file(os.path.join(ROOT, "scenes", "cornell.txt"), 800, 800).arrays, 800, 800, 64),
        "final": (final, 1200, 800, 100),
        "final+buried": (buried_light(final), 1200, 800, 100),
    }
    for name, (sc, *_) in scenes.items():  # one context per scene, so that the alternating steps do not re-upload
        ctxs[name] = Context(0)
        ctxs[name].set_scene(sc, use_bvh=True)
    dev, power_w, max_mhz = device_facts(ctxs["final"])
    rows = []
    for precision in ("f32", "f64"):
        dtype = np.float64 if precision == "f64" else np.float32
        for group in (["cornell"], ["final", "final+buried"]):
            rays, times, images = {}, {n: [] for n in group}, {}
            for n in group:
                _, W, H, spp = scenes[n]
                img, st = ctxs[n].render(W, H, spp, 50, seed=1984, count_rays=True, precision=precision, dtype=dtype)
                rays[n], images[n] = st["rays"], img
            for i in range(args.warmup + args.steps):
                for n in group:
                    _, W, H, spp = scenes[n]
                    img, st = ctxs[n].render(W, H, spp, 50, seed=1984, precision=precision, dtype=dtype)
                    if i >= args.warmup:
                        times[n].append(st["seconds_render"])
                    assert img.tobytes() == images[n].tobytes()
            if len(group) == 2:  # no path reaches the buried light: the same image and ray count as plain final.txt
                assert images["final"].tobytes() == images["final+buried"].tobytes() and rays["final"] == rays["final+buried"]
            for n in group:
                _, W, H, spp = scenes[n]
                t = np.array(times[n])
                row = dict(workload=n, precision=precision, W=W, H=H, spp=spp, depth=50, rays=int(rays[n]),
                           ms_median=float(np.median(t) * 1e3), ms_min=float(t.min() * 1e3), ms_max=float(t.max() * 1e3),
                           grays_per_s=float(rays[n] / np.median(t) * 1e-9), steps=args.steps, device=dev,
                           power_limit_w=power_w, max_sm_mhz=max_mhz)
                rows.append(row)
                print(json.dumps(row), flush=True)
    for c in ctxs.values():
        c.close()
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
