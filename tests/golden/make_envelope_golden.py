"""Generate tests/golden/reference_envelope.npz from the recorded runs of the UNMODIFIED reference EMD extension.

profiles/r2_s1_envelope.txt is the output of tools/envelope_probe.py on a B200: for the two batches of
test_emd_gpu.py::test_emd_deviation_lies_inside_the_reference_nondeterminism_envelope (bench.py's pool[0] and pool[1]:
table_clouds(32, 2048, seed=0), eps 0.005, 50 iterations) it ran the reference 12 times (4 repeats + 8 row orders) and
printed, per cloud, `ours - ref mean` and `ref std over 12` (numpy std, ddof=0) of the mean sqrt(dist).  `ours` there is
this package's kernel, which is bit-exact with oracle/emd_oracle.c (unchanged since before the recording), so the
reference's per-cloud mean is restored here as oracle - recorded difference; the recorded batch value of `ours` is checked
against the oracle first.  Usage: python tests/golden/make_envelope_golden.py
"""
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from pointcloud_b200 import synth  # noqa: E402


def _vector(text, label):
    m = re.search(re.escape(label) + r"\s*:\s*\[([^\]]*)\]", text)
    return np.array([float(v) for v in m.group(1).split()], np.float64)


def main():
    record = open(os.path.join(ROOT, "profiles", "r2_s1_envelope.txt")).read()
    out = {}
    for regime, block in zip(("independent", "noisy"), record.split("== ")[1:]):
        assert block.startswith(regime)
        x1, t = synth.table_clouds(32, 2048, seed=0, regime=regime)
        o = oracle.emd_forward(x1, t[:, :, :3].contiguous(), 0.005, 50, nthreads=os.cpu_count() or 1)
        ours = np.sqrt(o["dist"].astype(np.float64)).mean(1)
        recorded_batch = float(re.search(r"batch: ours (\S+)", block).group(1))
        assert abs(ours.mean() - recorded_batch) <= 1e-15, (ours.mean(), recorded_batch)
        races = np.array(json.loads(re.search(r"race events per cloud (\[[^\]]*\])", block).group(1)), np.int32)
        assert np.array_equal(races, o["race_events"])
        diff, std = _vector(block, "ours - ref mean"), _vector(block, "ref std over 12")
        assert diff.shape == std.shape == (32,)
        out[f"{regime}_ref_mean"] = ours - diff
        out[f"{regime}_ref_std"] = std * np.sqrt(12 / 11)         # ddof=1, as the live test computes it
        out[f"{regime}_race_events"] = races
    path = os.path.join(ROOT, "tests", "golden", "reference_envelope.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
