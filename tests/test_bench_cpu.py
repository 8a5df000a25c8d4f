"""bench.py contract checks that need no GPU: the reference arm (CPU oracle port) prints one JSON line with the keys
the driver reads, and the default arm refuses to run without a CUDA device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "clouds/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("chamfer+emd fwd+bwd clouds/sec") and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["vs_baseline"] is None and line["gpu_launches"] == 0 and "workload" in line["config"]


def test_steps_sets_the_timed_steps_and_bad_arguments_are_refused():
    run = lambda *a: subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *a], capture_output=True, text=True, timeout=600, cwd=ROOT)
    out = run("--impl", "reference", "--steps", "3", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = run(*bad)
        assert out.returncode == 2 and "error" in out.stderr, bad


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_default_arm_needs_a_gpu():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
