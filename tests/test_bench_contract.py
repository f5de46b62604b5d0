"""bench.py prints ONE JSON line with the keys the driver reads.  CPU: the reference arm (oracle/_ref/rrto or the
oracle port on the host cores).  GPU: our arm on a reduced spp (the headline config needs `python bench.py`)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
             "data", "config", "e2e", "gpu_launches"}


def run_bench(*args, timeout=900):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["unit"] == "Mrays/s" and d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_our_arm_line_reduced_spp():
    d = run_bench("--spp", "4", "--steps", "2", "--warmup", "3")
    assert BASE_KEYS | {"roofline", "cpu_baseline", "clocks", "kernel"} <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["scaling"] in ("weak", "strong")
    assert d["value"] > 100 and d["e2e"]["value"] > 100 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 1200 * 800 * 3 * 4
    assert d["gpu_launches"] == 4
    rf = d["roofline"]
    assert set(rf) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and 0 < rf["frac"] < 1.2 and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["value"] > 0 and cb["cores"] >= 1 and "sample" in cb
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_framebuffer_of_the_timed_path(tmp_path, ctx):
    """--dump-outputs writes the last timed step's framebuffer: the same sums the host-buffer render returns."""
    import numpy as np

    from conftest import load_golden

    d = run_bench("--spp", "4", "--steps", "2", "--warmup", "0", "--no-baselines", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    got = np.load(tmp_path / "image.npy")
    assert got.shape == (800, 1200, 3) and got.dtype == np.float32
    ctx.set_scene(load_golden("final")[0], use_bvh=True)
    want, _ = ctx.render(1200, 800, 4, 50, seed=1984)
    assert got.tobytes() == want.tobytes()
