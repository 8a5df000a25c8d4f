"""bench.py --dump-outputs: the files hold what the last timed step returned, on the inputs that step was given."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    steps, warmup = 6, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup), "--profile",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("losses", "grad_chamfer", "grad_emd")}
    assert all(a.dtype == np.float32 for a in got.values())

    import bench
    import pointcloud_b200 as pcl
    from pointcloud_b200 import synth
    last = warmup + steps - 1                                # the timed loop feeds pool[i % n_sets] for i in [warmup, warmup + steps)
    p, t, _ = bench.make_pool(torch, synth, torch.device("cuda", 0), 0, last + 1)[last]
    step = pcl.ShardedChamferEmdStep(bench.B_PER_GPU, bench.NPTS, torch.device("cuda", 0), bench.EPS, bench.ITERS)
    step.step(p, t)
    want = {"losses": step.out[:7], "grad_chamfer": step.grad_chamfer, "grad_emd": step.grad_emd}
    for n, w in want.items():
        assert got[n].shape == tuple(w.shape), n
        w = w.cpu().numpy()                                  # the Chamfer gradient is scattered with atomics: last-bit differences
        np.testing.assert_allclose(got[n], w, rtol=1e-5, atol=1e-7 * float(np.abs(w).max()), err_msg=n)
