"""bench.py's JSON contract on the arm that runs without a GPU: --impl reference (the CPU oracle), tiny workload."""
import json
import os
import subprocess
import sys

import numpy as np

import conftest


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(conftest.ROOT, "bench.py"), "--impl", "reference", "--small", "--width", "96",
                          "--height", "54", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=conftest.ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len(out.stdout.strip().splitlines()) == 1, "stdout carries the JSON line and nothing else"
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Mrays/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("Mrays/s") and line["value"] > 0 and line["steps"] == 2 and line["warmup"] == 1
    assert line["n_gpus"] == 1 and line["vs_baseline"] is None and line["data"] == "synthetic" and line["dtype"] == "f32"
    assert "workload" in line["config"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "96x54" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_reference_arm_dumps_the_last_step(tmp_path):
    outs = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(conftest.ROOT, "bench.py"), "--impl", "reference", "--small", "--width", "96",
                              "--height", "54", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=300, cwd=conftest.ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert os.listdir(tmp_path / run) == ["accumulation.npy"]
        outs.append(np.load(tmp_path / run / "accumulation.npy"))
    assert outs[0].dtype == np.float32 and outs[0].shape == (54, 96, 4)
    assert np.isfinite(outs[0]).all() and outs[0][..., :3].max() > 0
    assert np.array_equal(outs[0], outs[1])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(conftest.ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--small"],
                         capture_output=True, text=True, timeout=120, cwd=conftest.ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
