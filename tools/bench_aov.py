#!/usr/bin/env python
"""Cost of the first-hit AOV pass (rrtb_render_aov) next to the beauty render, one GPU.

    python tools/bench_aov.py [--steps K] [--warmup W] [--out FILE.jsonl]

Workloads, each in the float and the double integrator:
  final      final.txt 1200x800: the beauty render at 500 spp, depth 50 (the headline), and the AOV pass at 16, 64 and
             500 spp
  synthetic  BASELINE.json configs[4] (1 003 520 triangles + 100 004 spheres) at 3840x2160: the AOV pass at 64 spp and,
             as its yardstick, the beauty render at 64 spp, depth 50 (the config's 1024 spp would take 16 times as long)
Within a workload the renders alternate step by step.  Each row is the median device time (CUDA events) of K steps,
the primary segments per second (W x H x spp over that time; for the beauty render its camera paths) and the ratio to
the workload's beauty render.  The device name and power limit are read in the same run and printed with every row.
Writes nothing unless --out is given.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import load_workload  # noqa: E402
from bench_lights import device_facts  # noqa: E402
from rrt_b200 import Context  # noqa: E402

WORKLOADS = {  # name: (W, H, beauty spp, AOV spps)
    "final": (1200, 800, 500, (16, 64, 500)),
    "synthetic": (3840, 2160, 64, (64,)),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    rows = []
    dev = power_w = max_mhz = None
    for name, (W, H, beauty_spp, aov_spps) in WORKLOADS.items():
        scene, _ = load_workload(name, W, H)
        with Context(0) as ctx:
            ctx.set_scene(scene, use_bvh=True)
            if dev is None:
                dev, power_w, max_mhz = device_facts(ctx)
            for precision in ("f32", "f64"):
                dtype = np.float64 if precision == "f64" else np.float32
                runs = [("beauty", beauty_spp)] + [("aov", s) for s in aov_spps]
                times = {r: [] for r in runs}
                first = {}
                for i in range(args.warmup + args.steps):
                    for kind, spp in runs:
                        if kind == "beauty":
                            out, st = ctx.render(W, H, spp, 50, seed=1984, precision=precision, dtype=dtype)
                            blob = out.tobytes()
                        else:
                            out, st = ctx.render_aov(W, H, spp, seed=1984, precision=precision)
                            blob = b"".join(out[k].tobytes() for k in ("albedo", "normal", "depth", "coverage"))
                        assert first.setdefault((kind, spp), blob) == blob, "a repeat changed the output"
                        if i >= args.warmup:
                            times[(kind, spp)].append(st["seconds_render"])
                beauty_ms = float(np.median(times[runs[0]]) * 1e3)
                for kind, spp in runs:
                    t = np.array(times[(kind, spp)])
                    ms = float(np.median(t) * 1e3)
                    segments = W * H * spp  # the AOV pass: one primary segment per sample; the beauty render: its camera paths
                    row = {"workload": name, "pass": kind}
                    row.update(precision=precision, W=W, H=H, spp=spp,
                               depth=50 if kind == "beauty" else 1, ms_median=ms, ms_min=float(t.min() * 1e3),
                               ms_max=float(t.max() * 1e3), primary_segments_per_s=float(segments / (ms * 1e-3)),
                               ratio_to_beauty=ms / beauty_ms, beauty_spp=beauty_spp, steps=args.steps, device=dev,
                               power_limit_w=power_w, max_sm_mhz=max_mhz)
                    rows.append(row)
                    print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
