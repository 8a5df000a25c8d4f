"""The shared-memory poison helper of the stale-state tests builds for sm_100a without a GPU and exports both entry points."""
import ctypes
import subprocess

import smem_poison


def test_helper_builds_and_exports_poison_and_peek(tmp_path):
    so = smem_poison.build(str(tmp_path))
    syms = subprocess.run(["nm", "-D", "--defined-only", so], check=True, capture_output=True, text=True).stdout.split()
    assert "smem_poison" in syms and "smem_peek" in syms
    L = ctypes.CDLL(so)                     # loads without a device: nothing runs until a call
    assert L.smem_poison and L.smem_peek
