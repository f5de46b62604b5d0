#!/usr/bin/env python
"""bench.py -- the headline benchmark of the rrt hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes the framebuffer the last timed step produced (the [H, W, 3] sums of every pixel, row 0 =
bottom scanline, as rank 0 holds it) to DIR/image.npy, so that two builds run with the same arguments can be compared
output for output: the scene, the seed and therefore every sample are fixed by the arguments.  Over 64 MB, a fixed
sample of pixels is written with their indices (DIR/pixel_index.npy); --workload final_anim writes such a sample of
every frame of the animation, [frames, k, 3].

Workload (BASELINE.json configs[1]): scenes/final.txt (488 spheres), 1200x800, 500 spp, depth 50.
A step = one full render of that image: 480 M camera paths, ~1.21 G ray segments.
metric = Mrays/s = ray segments (closest-hit queries issued by the bounce loop) / seconds / 1e6.

  value     device-resident: scene + LBVH already in HBM; a step = zero accumulator + render kernel + the resolve
            epilogue (N > 1: every rank's epilogue stores its tiles as float3 into rank 0's frame over NVLink).
  e2e       through the reference-facing C ABI with HOST buffers: rrtb_scene_set (H2D scene + LBVH build)
            + rrtb_render (render + resolve + D2H framebuffer) inside the timed region, every step.
  roofline  FP32-issue roofline of the render kernel (SURVEY 8d): achieved = rays/s x W_ray lane-instr
            per ray (algorithmic count from the counting build's V_box, V_sph, ... on this very workload)
            against the issue rate MEASURED on this device by rrtb_probe_issue_rate.
  N > 1     the image is split by interleaved 8x4 tiles (strong scaling: total work fixed), one process per GPU;
            rank 0 owns the frame, the others map it once (CUDA IPC) and write their tiles into it from the resolve
            kernel (rrtb_render_shard): 12 B/pixel/N over NVLink, no reduce.  torch.distributed = handle + barriers.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, SPP, DEPTH, SEED = 1200, 800, 500, 50, 1984
METRIC = "Mrays/s on scenes/final.txt 1200x800 (500 spp, depth 50)"
UNIT = "Mrays/s"


WORKLOADS = {  # BASELINE.json configs[1..4]; configs[0] is the reference's own CPU case (a parity-test size)
    "final": dict(W=1200, H=800, spp=500, label="scenes/final.txt", config="BASELINE.json configs[1]", data="reference scene file scenes/final.txt"),
    "test3": dict(W=1920, H=1080, spp=256, label="scenes/test3.txt (motion blur)", config="BASELINE.json configs[2]", data="reference scene file scenes/test3.txt"),
    "test2": dict(W=1920, H=1080, spp=256, label="scenes/test2.txt (triangles)", config="BASELINE.json configs[3]", data="reference scene file scenes/test2.txt"),
    "final_anim": dict(W=1280, H=720, spp=50, label="scenes/final_anim (261 camera-only frames of final.txt)", config="SURVEY 8f2; reference scenes/final_anim/Makefile:9-10",
                       data="reference scene file scenes/final.txt + the camera path of scenes/final_anim/anim.py"),
    "synthetic": dict(W=3840, H=2160, spp=1024, label="synthetic 1 003 520 triangles + 100 004 spheres", config="BASELINE.json configs[4]",
                      data="synthetic scene generated in the reference grammar (rrt_b200/synthetic.py, seed 20221005)"),
    "synthetic_small": dict(W=3840, H=2160, spp=64, label="synthetic 250 880 triangles + 20 004 spheres", config="scaled-down sibling of configs[4]",
                            data="synthetic scene generated in the reference grammar (rrt_b200/synthetic.py, seed 20221005)"),
}


def load_workload(name, Wl, Hl):
    import tempfile

    import numpy as np

    from rrt_b200 import Scene, SceneArrays

    if name == "final" and (Wl, Hl) == (W, H):
        return final_scene()
    if name in ("final", "test2", "test3"):
        for base in (os.path.join(ROOT, "oracle", "_ref", "scenes"), "/root/reference/scenes"):
            p = os.path.join(base, name + ".txt")
            if os.path.exists(p):
                return Scene.from_file(p, Wl, Hl).arrays, p
        d = np.load(os.path.join(ROOT, "tests", "golden", "scene_%s.npz" % name))  # camera derived for the config's aspect
        return SceneArrays.from_npz_dict(d), "tests/golden/scene_%s.npz" % name
    from rrt_b200.synthetic import write_synthetic_scene

    kw = dict(n_spheres=100_000, ico_level=5, grid=7) if name == "synthetic" else dict(n_spheres=20_000, ico_level=4, grid=7)
    p = os.path.join(tempfile.gettempdir(), "rrtb_%s_%d.txt" % (name, os.getpid()))
    write_synthetic_scene(p, **kw)
    arrays = Scene.from_file(p, Wl, Hl).arrays
    os.remove(p)
    return arrays, "generated"


def final_scene():
    """scenes/final.txt.  Parsed by the product's own parser when the text is staged (oracle/_ref/scenes,
    which travels to the GPU box); otherwise the committed golden arrays, which are bit-identical to the
    parse (tests/test_host.py)."""
    import numpy as np

    from rrt_b200 import Scene, SceneArrays

    for p in (os.path.join(ROOT, "oracle", "_ref", "scenes", "final.txt"), "/root/reference/scenes/final.txt"):
        if os.path.exists(p):
            return Scene.from_file(p, W, H).arrays, p
    d = np.load(os.path.join(ROOT, "tests", "golden", "scene_final.npz"))
    return SceneArrays.from_npz_dict(d), "tests/golden/scene_final.npz"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 50 ms DURING the timed region.  The sampler is started before the
    warm-up steps (nvidia-smi needs a few hundred ms to produce its first line) and every line carries nvidia-smi's own
    timestamp; stop(t0, t1) keeps the samples taken inside the timed region [t0, t1] (wall-clock seconds), widened by one
    poll period on each side so that a region shorter than a poll still has its bracketing samples."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    POLL_MS = 50

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", str(self.POLL_MS)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    @staticmethod
    def _stamp(text):
        import datetime

        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(2 * self.POLL_MS * 1e-3)  # let the line that brackets the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        margin = self.POLL_MS * 1e-3
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            ts = self._stamp(f[0])
            if t0 is not None and ts is not None and not (t0 - margin <= ts <= t1 + margin):
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None,
                "poll_ms": self.POLL_MS, "lines_total": len(self.lines)}


# Algorithmic work per ray segment of each workload ON THE CANONICAL BINARY LBVH (the structure whose codes, order and
# topology are pinned bit-exactly against the oracle), measured once by the round-1 counting build
# (profiles/r01_bench_*.json).  The roofline numerator uses THIS figure, so that a better traversal structure (the
# 4-wide collapse, ...) raises the fraction instead of shrinking its own yardstick; the work actually traversed by the
# current structure is reported beside it as `w_ray_traversed`.
W_RAY_CANONICAL = {"final": 566.214, "synthetic": 1671.254, "test2": 293.815, "test3": 177.419}


def w_ray(st):
    """Algorithmic FP32 lane-instructions per ray segment (SURVEY 8d convention): ray setup 9, slab test 19,
    sphere 20, moving sphere 25, triangle 37, hit record 15 + scatter 80 on a hit, sky 15 on a miss."""
    r = float(st["rays"])
    vb, vs, vm, vt, h = (st[k] / r for k in ("box_tests", "sphere_tests", "msphere_tests", "triangle_tests", "hits"))
    return 9 + 19 * vb + 20 * vs + 25 * vm + 37 * vt + h * 95 + (1 - h) * 15, dict(V_box=vb, V_sph=vs, V_msph=vm, V_tri=vt, h=h)


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref/rrto = rrt.cpp
    built with -fopenmp, reference Makefile:45-46) on all host threads, on a bounded sample of the
    workload: the same scene and image at `REF_SPP` samples per pixel per step (cost is linear in spp).
    Falls back to the oracle port when the reference binary is absent."""
    if rank != 0:
        return
    import multiprocessing

    ref_spp = 2
    exe = os.path.join(ROOT, "oracle", "_ref", "rrto")
    scene_txt = os.path.join(ROOT, "oracle", "_ref", "scenes", "final.txt")
    cores = multiprocessing.cpu_count()
    # rays per camera path: a property of the estimator, measured by our counting build on this scene
    # (2.4913 at 1200x800; the reference's own instrumented value is 2.525, SURVEY Appendix C)
    rays_per_path = 2.4913
    try:
        with open(os.path.join(ROOT, "profiles", "workload_final.json")) as f:
            rays_per_path = json.load(f)["rays_per_path"]
    except Exception:
        pass
    times = []
    kind = "reference"
    if os.path.exists(exe) and os.path.exists(scene_txt):
        for i in range(args.warmup + args.steps):
            r = subprocess.run([exe, "-i", scene_txt, "-w", str(W), "-h", str(H), "-s", str(ref_spp), "-d", str(DEPTH), "-o", "/tmp/_rrto.png"],
                               capture_output=True, text=True)
            sec = None
            for ln in r.stderr.splitlines():
                if ln.startswith("stats,"):
                    sec = float(ln.split(",")[-1])
            if sec is None:
                raise RuntimeError("rrto produced no stats line: " + r.stderr[-300:])
            if i >= args.warmup:
                times.append(sec)
        sample = "oracle/_ref/rrto (reference rrt.cpp, OpenMP double) final.txt %dx%d at %d spp per step" % (W, H, ref_spp)
    else:
        kind = "port"
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from oracle_lib import Oracle

        scene, _ = final_scene()
        orc = Oracle(scene)
        for i in range(args.warmup + args.steps):
            t0 = time.time()
            _, _, cnt = orc.render(W, H, ref_spp, DEPTH, SEED)
            if i >= args.warmup:
                times.append(time.time() - t0)
        rays_per_path = cnt["rays"] / cnt["paths"]
        sample = "oracle port (rrt_oracle.c, OpenMP) final.txt %dx%d at %d spp per step" % (W, H, ref_spp)
    sec = sum(times) / len(times)
    value = W * H * ref_spp * rays_per_path / sec / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "reference scene file scenes/final.txt",
        "config": {"workload": "scenes/final.txt 1200x800 depth 50, bounded sample: %d spp per step" % ref_spp, "rays_per_path": rays_per_path},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_gpu_baseline(spp=50):
    """The reference's own rrt.cu rebuilt for sm_100a (oracle/_ref/rrt), timed in the same run on the same scene: the
    block shapes of BASELINE.md section 3 (the reference's PERFORMANCE.txt:6-19 has wide flat blocks as its fastest)
    at a bounded spp (its cost is linear in spp), then the best shape once at the full 500 spp.  Not an optimisation
    target."""
    exe = os.path.join(ROOT, "oracle", "_ref", "rrt")
    scene_txt = os.path.join(ROOT, "oracle", "_ref", "scenes", "final.txt")
    if not (os.path.exists(exe) and os.path.exists(scene_txt)):
        return None

    def run(tx, ty, n_spp):
        try:
            r = subprocess.run([exe, "-i", scene_txt, "-w", str(W), "-h", str(H), "-s", str(n_spp), "-d", str(DEPTH), "-tx", str(tx), "-ty", str(ty), "-o", "/tmp/_rrt_ref.png"],
                               capture_output=True, text=True, timeout=600)
        except Exception:
            return None
        for ln in r.stderr.splitlines():
            if ln.startswith("stats,"):
                return float(ln.split(",")[-1])
        return None

    sweep = {}
    for tx, ty in ((8, 8), (16, 16), (128, 2), (256, 1), (512, 1)):
        sec = run(tx, ty, spp)
        if sec is not None:
            sweep["%dx%d" % (tx, ty)] = sec
    if not sweep:
        return None
    block = min(sweep, key=sweep.get)
    out = {"seconds": sweep[block], "spp": spp, "block": block, "sweep_seconds_at_%d_spp" % spp: sweep}
    tx, ty = (int(x) for x in block.split("x"))
    full = run(tx, ty, SPP)
    if full is not None:
        out["seconds_at_500_spp"] = full
    return out


def cpu_baseline_sample(rays_per_path):
    """rank 0, N=1 only: the reference CPU path (rrto) on a bounded sample, on the box's host cores."""
    import multiprocessing

    exe = os.path.join(ROOT, "oracle", "_ref", "rrto")
    scene_txt = os.path.join(ROOT, "oracle", "_ref", "scenes", "final.txt")
    cores = multiprocessing.cpu_count()
    spp = 4
    if os.path.exists(exe) and os.path.exists(scene_txt):
        r = subprocess.run([exe, "-i", scene_txt, "-w", str(W), "-h", str(H), "-s", str(spp), "-d", str(DEPTH), "-o", "/tmp/_rrto.png"],
                           capture_output=True, text=True)
        for ln in r.stderr.splitlines():
            if ln.startswith("stats,"):
                f = ln.split(",")
                sec, threads = float(f[-1]), int(f[-4])
                return {"value": W * H * spp * rays_per_path / sec / 1e6, "unit": UNIT, "cores": threads, "kind": "reference",
                        "sample": "oracle/_ref/rrto (reference rrt.cpp, OpenMP, double) final.txt %dx%d, %d spp, %.2f s" % (W, H, spp, sec)}
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle

    scene, _ = final_scene()
    t0 = time.time()
    _, _, cnt = Oracle(scene).render(W, H, spp, DEPTH, SEED)
    sec = time.time() - t0
    return {"value": cnt["rays"] / sec / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "oracle port (OpenMP) final.txt %dx%d, %d spp, %.2f s" % (W, H, spp, sec)}


DUMP_BYTES = 64 * 10**6  # every file of one dump together, .npy headers included
DUMP_SAMPLE_PIXELS = 1 << 20


def dump_pixel_sample(n_pixels, k):
    """k of n_pixels flat pixel indices, sorted; seeded, so the same for every run of the same image size."""
    import numpy as np

    return np.sort(np.random.default_rng(SEED).choice(n_pixels, k, replace=False))


def dump_outputs(dirname, image, pixel_index=None):
    """DIR/image.npy = the [H, W, 3] framebuffer.  A framebuffer larger than DUMP_BYTES is replaced by a fixed sample of
    DUMP_SAMPLE_PIXELS pixels: DIR/image.npy holds their [k, 3] sums and DIR/pixel_index.npy their flat indices y * W + x.
    A caller that sampled the pixels itself passes their indices as pixel_index."""
    import numpy as np

    os.makedirs(dirname, exist_ok=True)
    image = np.asarray(image)
    assert image.dtype in (np.float32, np.float64)
    if pixel_index is None and image.nbytes > DUMP_BYTES:
        px = image.reshape(-1, 3)
        pixel_index = dump_pixel_sample(len(px), DUMP_SAMPLE_PIXELS)
        image = px[pixel_index]
    if pixel_index is not None:
        np.save(os.path.join(dirname, "pixel_index.npy"), np.asarray(pixel_index).astype(np.float64))
    np.save(os.path.join(dirname, "image.npy"), image)


def run_anim(args, wl, rank, world, local_rank):
    """--workload final_anim: the reference's 261-frame camera dolly (1280x720, 50 spp) as ONE uploaded scene +
    one camera update and one kernel launch per frame; frames dealt round-robin over the ranks (no collective).
    A step = the whole animation."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from rrt_b200 import Context
    from rrt_b200.anim import final_anim_cameras, frames_of_rank

    Wl, Hl, spp = args.width or wl["W"], args.height or wl["H"], (args.spp if args.spp != SPP else wl["spp"])
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(local_rank)
    scene, src = load_workload("final", Wl, Hl)
    cams = final_anim_cameras(Wl, Hl)
    mine = frames_of_rank(len(cams), rank, world)
    ctx = Context(local_rank)
    ctx.set_scene(scene, use_bvh=True)
    n = 3 * Wl * Hl
    acc = torch.zeros(n, dtype=torch.int64, device=dev)
    out = torch.empty(n, dtype=torch.float32, device=dev)
    host = np.empty((Hl, Wl, 3), np.float32)
    params = ctx.params(Wl, Hl, spp, DEPTH, SEED)
    pcount = ctx.params(Wl, Hl, spp, DEPTH, SEED, count_rays=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(p=params, keep=None):
        rays = 0
        for f in mine:
            ctx.set_camera(cams[f])
            acc.zero_()
            torch.cuda.synchronize()
            st = ctx.render_device(p, acc.data_ptr())
            rays += st["rays"]
            ctx.resolve_device(acc.data_ptr(), out.data_ptr(), n)
            if keep is not None:
                keep[f] = out.view(-1, 3)[keep_index]
        return rays

    rays = torch.tensor([step(pcount)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(rays)
    total_rays = int(rays.item())
    for _ in range(max(args.warmup - 1, 0)):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1) * 1e-3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = t.item() / args.steps
    if args.dump_outputs:
        # a step renders every frame, each into the same buffer: the last step is rendered once more, untimed (same
        # cameras, same seed, hence the same sums), keeping a fixed pixel sample of every frame, gathered on rank 0
        k = min(Wl * Hl, (DUMP_BYTES - 4096) // (12 * len(cams) + 8))  # float3 per frame + a float64 index per pixel
        idx = dump_pixel_sample(Wl * Hl, k)
        keep_index = torch.from_numpy(idx).to(dev)
        frames = torch.zeros((len(cams), k, 3), dtype=torch.float32, device=dev)
        step(keep=frames)
        if world > 1:
            dist.all_reduce(frames)  # every frame is rendered by one rank; the others contribute zeros
        if rank == 0:
            frames = frames.cpu().numpy()
            if k == Wl * Hl:
                dump_outputs(args.dump_outputs, frames.reshape(len(cams), Hl, Wl, 3))
            else:
                dump_outputs(args.dump_outputs, frames, idx)
    # e2e: host framebuffer per frame through rrtb_render (D2H inside), scene uploaded once per step
    barrier()
    t0 = time.perf_counter()
    ctx.set_scene(scene, use_bvh=True)
    for f in mine:
        ctx.set_camera(cams[f])
        ctx.render(Wl, Hl, spp, DEPTH, SEED, out=host)
    barrier()
    e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e, op=dist.ReduceOp.MAX)
    if rank == 0:
        line = {
            "metric": "Mrays/s on %s" % wl["label"], "value": total_rays / sec / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 (f64 leaf discriminants, u64 fixed-point accumulation)", "data": "%s (%s)" % (wl["data"], src),
            "config": {"workload": "%s %dx%d, %d spp, depth 50 (%s)" % (wl["label"], Wl, Hl, spp, wl["config"]), "frames": len(cams),
                       "frames_per_s": len(cams) / sec, "sharding": "frames round-robin over %d GPU(s), no collective" % world,
                       "rays_per_step": total_rays, "reference": "README of scenes/final_anim: 3.3 hours for the same 261 frames (author's GPU)"},
            "e2e": {"value": total_rays / e.item() / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(scene.spheres.nbytes + scene.materials.nbytes + 96 * len(cams)),
                    "d2h_bytes_per_step": int(host.nbytes * len(cams)), "seconds_per_animation": e.item()},
            "gpu_launches": args.steps * 2 * len(cams),
        }
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--spp", type=int, default=SPP, help="debug only: any value other than 500 is not the headline config")
    ap.add_argument("--no-baselines", action="store_true", help="skip the cpu / reference-GPU baselines (profiling runs)")
    ap.add_argument("--workload", default="final", choices=sorted(WORKLOADS), help="final = the headline (BASELINE.json configs[1]); the others are the remaining configs")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--shard", default="tiles", choices=["tiles", "samples"])
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"], help="f64 = the double integrator (the reference's rrtd build); not the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the framebuffer of the last timed step to DIR/image.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computed")

    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # `python bench.py --gpus N` without a launcher: re-run under torch.distributed.run, one rank per GPU
        import socket

        with socket.socket() as so:
            so.bind(("127.0.0.1", 0))
            port = so.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from rrt_b200 import Context

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.workload == "final_anim":
        return run_anim(args, WORKLOADS[args.workload], rank, world, local_rank)
    wl = WORKLOADS[args.workload]
    Wl, Hl = args.width or wl["W"], args.height or wl["H"]
    spp = args.spp if (args.spp != SPP or args.workload == "final") else wl["spp"]
    headline = args.workload == "final" and spp == SPP and (Wl, Hl) == (W, H)
    shard_mode = 0 if args.shard == "tiles" else 1

    scene, scene_src = load_workload(args.workload, Wl, Hl)
    ctx = Context(local_rank)
    ctx.set_scene(scene, use_bvh=True)
    n = 3 * Wl * Hl
    acc = torch.zeros(n, dtype=torch.int64, device=dev)
    out = torch.empty(n, dtype=torch.float32, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2
    f64 = args.precision == "f64"
    headline = headline and not f64
    params = ctx.params(Wl, Hl, spp, DEPTH, SEED, rank, world, shard_mode, False, precision=args.precision)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    kernel_seconds = []

    dr = None
    if world > 1:  # rank 0 owns the frame, the others map it (CUDA IPC); see rrt_b200/dist.py
        from rrt_b200.dist import DistributedRenderer

        dr = DistributedRenderer(ctx, rank, world)
        dr.ensure_frame(Wl, Hl, f64)

    def step():
        flush.fill_(1.0)  # L2 flush between timed iterations (the scene itself is far smaller than L2)
        if world == 1:
            acc.zero_()
            torch.cuda.synchronize()  # ctx renders on its own stream
            st = ctx.render_device(params, acc.data_ptr())
            ctx.resolve_device(acc.data_ptr(), out.data_ptr(), n)
        else:
            torch.cuda.synchronize()
            st = ctx.render_shard(params)  # zero own accumulator + render + epilogue into rank 0's frame over NVLink
        kernel_seconds.append(st["seconds_render"])

    # counting pass (untimed): rays and per-ray work of exactly this workload and shard
    pc = ctx.params(Wl, Hl, spp, DEPTH, SEED, rank, world, shard_mode, True, precision=args.precision)
    acc.zero_()
    torch.cuda.synchronize()
    cst = ctx.render_device(pc, acc.data_ptr())
    counts = torch.tensor([cst[k] for k in ("rays", "box_tests", "sphere_tests", "msphere_tests", "triangle_tests", "hits", "paths")],
                          dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(counts)
    tot = dict(zip(("rays", "box_tests", "sphere_tests", "msphere_tests", "triangle_tests", "hits", "paths"), counts.tolist()))
    total_rays = tot["rays"]

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # before the warm-up: nvidia-smi is up and printing by the time the timed region starts
    for _ in range(args.warmup):
        step()
    kernel_seconds.clear()
    barrier()
    wall0 = time.time()
    t0 = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    dev_s = ev0.elapsed_time(ev1) * 1e-3
    clocks = sampler.stop(wall0, wall0 + wall) if rank == 0 else None
    # max over ranks of the device-timed region
    tt = torch.tensor([dev_s, wall, sum(kernel_seconds) / len(kernel_seconds)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_s, wall, kern_s = tt.tolist()
    sec_per_step = dev_s / args.steps
    value = total_rays / sec_per_step / 1e6
    if args.dump_outputs:
        image = np.empty((Hl, Wl, 3), np.float64 if f64 else np.float32) if rank == 0 else None
        if world > 1 and shard_mode == 1:
            # the ranks ADD their samples into rank 0's sum buffer, which only a download resolves and clears: it holds
            # every step so far.  Clear it, then render the last step once more, untimed (same seed, same sums).
            if rank == 0:
                ctx.frame_download(image, shard_mode)
            barrier()
            step()
            barrier()
        if rank == 0:
            # world > 1, tiles: every rank's tiles of the last step are in rank 0's frame (barrier above)
            image = out.cpu().numpy().reshape(Hl, Wl, 3) if world == 1 else ctx.frame_download(image, shard_mode)
            dump_outputs(args.dump_outputs, image)

    # ---- e2e: through the C ABI with HOST buffers, every step: scene upload + LBVH build + render + D2H of the frame
    from rrt_b200 import PinnedBuffer

    pin = PinnedBuffer((Hl, Wl, 3), np.float64 if f64 else np.float32) if rank == 0 else None  # pinned: the D2H is one DMA
    host_out = pin.array if rank == 0 else None
    h2d = scene.camera.nbytes + scene.materials.nbytes + scene.spheres.nbytes + scene.mspheres.nbytes + scene.triangles.nbytes
    d2h = host_out.nbytes if rank == 0 else 0

    def e2e_step():
        if world == 1:
            ctx.set_scene(scene, use_bvh=True)
            ctx.render(Wl, Hl, spp, DEPTH, SEED, out=host_out, precision=args.precision)
        else:
            dist.barrier()  # rank 0 has read the previous frame
            ctx.set_scene(scene, use_bvh=True)
            ctx.render_shard(params)
            dist.barrier()  # every rank's tiles are in rank 0's frame
            if rank == 0:
                ctx.frame_download(host_out, shard_mode)

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = total_rays / (e2e_t.item() / e2e_steps) / 1e6

    if rank == 0:
        wr_trav, v = w_ray(tot)
        wr = W_RAY_CANONICAL.get(args.workload, wr_trav) if (Wl, Hl) == (wl["W"], wl["H"]) else wr_trav
        probe = ctx.probe_issue_rate()
        info = ctx.device_info()
        nominal = info["sm_count"] * 128 * info["clock_khz"] * 1e3  # lanes x clock: 1 warp-instruction / clk / SM sub-partition
        kern_rays_per_s = (cst["rays"] if world == 1 else tot["rays"] / world) / kern_s
        achieved = kern_rays_per_s * wr  # lane-instr / s, per GPU
        peak = max(probe["ffma"], probe["ffma_fmnmx_mix"])  # the issue-rate ceiling: 1 warp-instr / clk / SMSP
        traffic = None  # dram bytes per launch of the render kernel, from the committed ncu --set full capture
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                traffic = json.load(f)["traffic_bytes_per_launch"] if (headline and world == 1) else None
        except Exception:
            pass
        line = {
            "metric": (METRIC if args.workload == "final" else "Mrays/s on %s" % wl["label"]) + (" [double integrator, rrtd semantics]" if f64 else ""), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64 (float slab tests, u64 fixed-point accumulation)" if f64 else "f32 (f64 leaf discriminants, u64 fixed-point accumulation)",
            "data": "%s (%s)" % (wl["data"], scene_src),
            "config": {"workload": "%s %dx%d, %d spp, depth 50 (%s)" % (wl["label"], Wl, Hl, spp, wl["config"]), "prims": scene.n_objects,
                       "sharding": "one image, %s over %d GPU(s); %s" % ("interleaved 8x4 tiles" if shard_mode == 0 else "interleaved samples", world,
                                                                         "single GPU" if world == 1 else ("each rank's resolve kernel stores its tiles as float3 into rank 0's frame over NVLink (CUDA IPC peer mapping): %d bytes per frame cross the link" % (12 * Wl * Hl * (world - 1) // world) if shard_mode == 0 else "each rank adds its u64 partial sums into rank 0's buffer over NVLink (integer atomics)")),
                       "l2": "256 MiB flush written between timed iterations", "rays_per_step": total_rays,
                       "rays_per_path": total_rays / tot["paths"], **{k: round(x, 4) for k, x in v.items()}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "what": "rrtb_scene_set (upload + LBVH build + 4-wide collapse) + " + ("rrtb_render (render + resolve + D2H into pinned host memory)" if world == 1 else "rrtb_render_shard on every rank + 2 barriers + rrtb_frame_download on rank 0 (pinned host memory)") + " per step"},
            "gpu_launches": args.steps * 2,
            "kernel": {"name": "rrtb::k_render_pool<false,2,true,PathF64>" if f64 else "rrtb::k_render_pool<false,2,false,PathF32>", "avg_ms": kern_s * 1e3, "share_of_step": kern_s / sec_per_step},
            "roofline": {"bound": "fp32_issue", "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "T lane-instr/s",
                         "frac": achieved / peak, "frac_nominal": achieved / nominal, "peak_nominal": nominal / 1e12, "traffic": traffic, "w_ray": wr,
                         "w_ray_traversed": wr_trav,
                         "w_ray_note": "w_ray = algorithmic lane-instructions per ray segment on the canonical binary LBVH (round-1 counting build, fixed per workload); w_ray_traversed = the same cost model over what the current 4-wide tree visits",
                         "peak_source": "measured on this device by rrtb_probe_issue_rate: FFMA-only loop %.2f T lane-instr/s (an FFMA+FMNMX "
                                        "slab-test mix reaches %.2f); nominal 148 SM x 128 lanes x 1.965 GHz = 37.2; MEASURED_PEAKS.json "
                                        "has no FP32 figure" % (probe["ffma"] / 1e12, probe["ffma_fmnmx_mix"] / 1e12),
                         "hbm_note": "scene + LBVH = %d KB (L1/L2 resident); HBM traffic is the %d MB u64 accumulator" % ((scene.n_objects * (64 + 48 + 8)) // 1024, n * 8 // 2**20)},
            "clocks": clocks,
            "wall_s": wall,
        }
        if f64:
            line["roofline"]["note"] = "W_ray counts the float integrator's instructions; reported for throughput only in the f64 build"
        if world == 1 and not args.no_baselines and args.workload == "final" and not f64:
            line["cpu_baseline"] = cpu_baseline_sample(total_rays / tot["paths"])
            g = reference_gpu_baseline()
            if g:
                g["Mrays/s"] = W * H * g["spp"] * (total_rays / tot["paths"]) / g["seconds"] / 1e6
                if "seconds_at_500_spp" in g:
                    g["Mrays/s_at_500_spp"] = W * H * SPP * (total_rays / tot["paths"]) / g["seconds_at_500_spp"] / 1e6
                g["what"] = "reference rrt.cu rebuilt for sm_100a (oracle/_ref/rrt), float, its own BVH, best of 5 block shapes at 50 spp, then that shape at 500 spp"
                line["reference_gpu"] = g
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
