"""Shared-memory poison and canary (tests/smem_poison.cu).  TEST INFRASTRUCTURE ONLY.  The CUDA file is compiled on first
use into a private temporary directory (the tree may be read-only) with the nvcc of pointcloud_b200/build.py, for sm_100a."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
MAX_SMID = 1024          # length of the per-%smid counters
_lib = None


def build(outdir):
    """Compile tests/smem_poison.cu into outdir/libsmem_poison.so and return its path (needs nvcc, no GPU)."""
    from pointcloud_b200 import build as B
    so = os.path.join(outdir, "libsmem_poison.so")
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.run([B._nvcc(), "-ccbin", ccbin, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared",
                    "-Xcompiler", "-fPIC", "-o", so, os.path.join(_HERE, "smem_poison.cu")], check=True)
    return so


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="smem_poison_")
        atexit.register(shutil.rmtree, d, True)
        L = ctypes.CDLL(build(d))
        L.smem_poison.restype = ctypes.c_int
        L.smem_poison.argtypes = [ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.smem_peek.restype = ctypes.c_int
        L.smem_peek.argtypes = [ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib = L
    return _lib


def _ctas():
    import torch
    return 4 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def poison(pattern, stream, sm_hits):
    """Fill the shared memory of every SM with the 32-bit `pattern`, on `stream` (a torch.cuda.Stream); sm_hits is a zeroed
    int32 CUDA tensor of MAX_SMID entries that receives the number of poison CTAs per %smid."""
    rc = lib().smem_poison(pattern & 0xFFFFFFFF, _ctas(), sm_hits.data_ptr(), stream.cuda_stream)
    assert rc == 0, f"smem_poison failed ({rc})"


def peek(pattern, stream, sm_hits, sm_bad):
    """The canary: sm_hits / sm_bad (zeroed int32 CUDA tensors of MAX_SMID entries) receive, per %smid, the CTAs that ran
    there and those that found a shared-memory word other than `pattern`."""
    rc = lib().smem_peek(pattern & 0xFFFFFFFF, _ctas(), sm_hits.data_ptr(), sm_bad.data_ptr(), stream.cuda_stream)
    assert rc == 0, f"smem_peek failed ({rc})"
