"""bench.py's reference arm runs without a GPU and prints ONE JSON line with the contract's keys; on a GPU (-m gpu), --steps sets
the timed steps and --dump-outputs writes the last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gaussians", "5000", "--width", "160",
                        "--height", "96", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Mpix/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and "workload" in d["config"]


def test_non_rank0_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--gaussians", "100",
                        "--width", "32", "--height", "32", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120,
                       cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    P, V, steps = 100_000, 2, 3
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gaussians", str(P), "--width", "160", "--height", "96",
                        "--views-per-rank", str(V), "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
    assert d["steps"] == steps and d["single_view"]["views_timed"] == steps * V
    inputs = ("means3D", "shs", "opacities", "scales", "rotations")
    arrays = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(arrays) == {"gaussian_index", "losses", "radii_max"} | {"grad_" + n for n in inputs}
    assert sum(os.path.getsize(out / (k + ".npy")) for k in arrays) <= 64 << 20
    idx = arrays.pop("gaussian_index")
    assert idx.dtype == np.float64 and idx.shape == (65536,) and (np.diff(idx) > 0).all() and 0 <= idx[0] and idx[-1] < P
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert arrays["losses"].shape == (V,) and (arrays["losses"] > 0).all()
    assert (arrays["radii_max"] >= 0).all() and (arrays["radii_max"] > 0).any()
    shapes = {"means3D": (3,), "shs": (16, 3), "opacities": (1,), "scales": (3,), "rotations": (4,)}
    for n in inputs:
        g = arrays["grad_" + n]
        assert g.shape == (65536, *shapes[n]) and np.abs(g).max() > 0, n
        # a gaussian no view saw has no gradient
        assert not np.abs(g[arrays["radii_max"] == 0]).any(), n
