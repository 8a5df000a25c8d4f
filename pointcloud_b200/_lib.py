"""ctypes loader for libpcl_b200.so (the C ABI declared in include/pcl.h).

There is no fallback of any kind: if the library is missing it is built with nvcc; if that fails, or
if a compute entry point is called without a CUDA device, an exception is raised.
"""
import ctypes
import os

import torch

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

PCL_F32, PCL_F16, PCL_BF16 = 0, 1, 2
PCL_CHAMFER_UNFUSED, PCL_CHAMFER_FMA = 0, 1
_DTYPES = {torch.float32: PCL_F32, torch.float16: PCL_F16, torch.bfloat16: PCL_BF16}

c_void_p, c_int, c_int64, c_size_t, c_float = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float
c_double = ctypes.c_double

_PTS = [c_void_p, c_int, c_int64, c_int64]  # pointer, dtype, batch stride, row stride
_SIGNATURES = {
    "pcl_version": (c_int, []),
    "pcl_last_error": (ctypes.c_char_p, []),
    "pcl_device_info": (c_int, [ctypes.POINTER(c_int)] * 4),
    "pcl_chamfer_set_prune_min": (c_int, [c_int]),
    "pcl_chamfer_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pcl_chamfer_fwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 5 + [c_void_p] * 5 + [c_void_p, c_size_t, c_void_p]),
    "pcl_chamfer_bwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 4 + [c_void_p] * 5 + [c_void_p]),
    "pcl_chamfer_cloud_fwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 5 + [c_void_p] * 6 + _PTS + _PTS + [c_void_p]
                              + [c_void_p, c_size_t, c_void_p]),
    "pcl_chamfer_cloud_bwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 4 + [c_void_p] * 5 + _PTS + _PTS + [c_void_p] * 3
                              + [c_void_p]),
    "pcl_emd_max_points": (c_int, []),
    "pcl_emd_set_path": (c_int, [c_int]),
    "pcl_emd_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pcl_emd_fwd": (c_int, _PTS + _PTS + [c_int, c_int, c_float, c_int] + [c_void_p] * 3 + [c_void_p, c_size_t, c_void_p]),
    "pcl_emd_fwd_fused": (c_int, _PTS + _PTS + [c_int, c_int, c_float, c_int] + [c_void_p] * 3 + [c_float, c_void_p, c_void_p] + [c_void_p, c_size_t, c_void_p]),
    "pcl_emd_bwd": (c_int, _PTS + _PTS + [c_int, c_int] + [c_void_p] * 3 + [c_void_p]),
    "pcl_emd_match_hist": (c_int, _PTS + [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "pcl_emd_weighted_reduce": (c_int, [c_void_p] * 3 + [c_int] * 3 + [c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcl_emd_weighted_bwd": (c_int, _PTS + _PTS + [c_int, c_int] + [c_void_p] * 4 + [c_int] + [c_void_p] * 3 + [c_void_p]),
    "pcl_emd_feature_workspace_bytes": (c_size_t, []),
    "pcl_emd_seg_ce_fwd": (c_int, _PTS + [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcl_emd_seg_ce_bwd": (c_int, _PTS + [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "pcl_emd_feat_mse_fwd": (c_int, _PTS + _PTS + [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "pcl_emd_feat_mse_bwd": (c_int, _PTS + _PTS + [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "pcl_class_filter": (c_int, _PTS + [c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "pcl_fps_max_points": (c_int, []),
    "pcl_fps": (c_int, _PTS + [c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "pcl_fps_ragged": (c_int, _PTS + [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "pcl_ball_query": (c_int, _PTS + _PTS + [c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p]),
    "pcl_knn_max_k": (c_int, []),
    "pcl_knn_fwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 6 + [c_void_p] * 2 + [c_void_p]),
    "pcl_knn_bwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 5 + [c_void_p] * 4 + [c_void_p]),
    "pcl_ball_query_fwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 5 + [c_float, c_int] + [c_void_p] * 2 + [c_void_p]),
    "pcl_ball_query_bwd": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 5 + [c_void_p] * 4 + [c_void_p]),
    "pcl_frames_fwd": (c_int, _PTS + [c_void_p] + [c_int] * 4 + [c_void_p] * 3 + [c_void_p]),
    "pcl_frames_bwd": (c_int, _PTS + [c_void_p] + [c_int] * 3 + [c_void_p] * 6 + [c_void_p]),
    "pcl_points_alignment_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pcl_points_alignment_fwd": (c_int, _PTS + _PTS + [c_void_p] * 2 + [c_int] * 4 + [c_double] + [c_void_p] * 4 + [c_void_p, c_size_t, c_void_p]),
    "pcl_points_alignment_bwd": (c_int, _PTS + _PTS + [c_void_p] * 2 + [c_int] * 3 + [c_double] + [c_void_p] * 7 + [c_void_p]),
    "pcl_icp_workspace_bytes": (c_size_t, [c_int] * 4),
    "pcl_icp": (c_int, _PTS + [c_void_p] + _PTS + [c_void_p] + [c_int] * 3 + [c_void_p] * 3 + [c_int, c_float, c_int, c_int, c_int]
                + [c_void_p] * 6 + [c_void_p, c_size_t, c_void_p]),
    "pcl_points_to_volumes_fwd": (c_int, _PTS + _PTS + [c_void_p] * 2 + [c_int] * 8 + [c_void_p] * 2 + [c_void_p]),
    "pcl_points_to_volumes_bwd": (c_int, _PTS + _PTS + [c_void_p] * 2 + [c_int] * 8 + [c_void_p] * 4 + [c_void_p]),
    "pcl_raster_max_k": (c_int, []),
    "pcl_rasterize_points_workspace_bytes": (c_size_t, [c_int] * 6),
    "pcl_rasterize_points_fwd": (c_int, _PTS + [c_void_p, c_void_p, c_float] + [c_int] * 7 + [c_void_p] * 3 + [c_void_p, c_size_t, c_void_p]),
    "pcl_rasterize_points_bwd": (c_int, _PTS + [c_void_p] + [c_int] * 5 + [c_void_p] * 4 + [c_void_p]),
    "pcl_composite_fwd": (c_int, [c_int, c_void_p, c_int] + [c_void_p] * 5 + [c_int] * 5 + [c_int64, c_void_p, c_void_p]),
    "pcl_composite_bwd": (c_int, [c_int, c_void_p, c_int] + [c_void_p] * 5 + [c_int] * 5 + [c_int64] + [c_void_p] * 4),
    "pcl_chamfer_emd_step_scratch_bytes":(c_size_t, [c_int, c_int]),
    "pcl_chamfer_emd_step": (c_int, _PTS + _PTS + [c_int, c_int, c_float, c_int, c_int] + [c_void_p] * 3 + [c_void_p, c_size_t, c_void_p]),
    "pcl_loss_host_scratch_bytes": (c_size_t, [c_int, c_int]),
    "pcl_chamfer_emd_step_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_int] + [c_void_p] * 3 + [c_void_p, c_size_t, c_void_p]),
}


class PclError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.LIB


def lib():
    """Load (building first if necessary) the CUDA library.  Raises if it cannot be had."""
    global _LIB
    if _LIB is None:
        path = _build.build()
        L = ctypes.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if include/pcl.h and the library disagree
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


def check(rc: int, what: str):
    if rc != 0:
        raise PclError(f"{what} failed (code {rc}): {lib().pcl_last_error().decode()}")


_HAVE_CUDA = None


def require_cuda():
    global _HAVE_CUDA
    if _HAVE_CUDA is None:
        _HAVE_CUDA = bool(torch.cuda.is_available())
    if not _HAVE_CUDA:
        raise PclError("pointcloud_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def stream_ptr(device=None) -> int:
    """Raw cudaStream_t of torch's current stream on `device` (default: the current device) -- the C-level accessor, a
    fraction of a microsecond, where torch.cuda.current_stream().cuda_stream builds a Stream object (~20 us)."""
    idx = device.index if (device is not None and device.index is not None) else torch.cuda.current_device()
    return torch._C._cuda_getCurrentRawStream(idx)


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NO_GUARD = _NoGuard()


def on_device(device):
    """Device guard that costs nothing when `device` already is the current device (the one-rank-one-device case)."""
    if device.index is None or device.index == torch.cuda.current_device():
        return _NO_GUARD
    return torch.cuda.device(device)


def pts_args(t: torch.Tensor):
    """(ptr, dtype, batch stride, row stride) of a (B,P,D) CUDA tensor view with unit channel stride."""
    assert t.dim() == 3 and t.is_cuda
    return [t.data_ptr(), _DTYPES[t.dtype], t.stride(0), t.stride(1)]


def as_points(t: torch.Tensor) -> torch.Tensor:
    """Make a tensor usable by the kernels WITHOUT copying whenever it already is a CUDA
    fp32/fp16/bf16 view with unit channel stride (e.g. pred[:, :, :3]); otherwise mirror the
    reference's `.contiguous().float().cuda()` (emd_module.py:43-44)."""
    if not t.is_cuda:
        require_cuda()
        t = t.cuda()
    if t.dtype not in _DTYPES:
        t = t.float()
    if t.dim() != 3:
        raise ValueError(f"expected a (B, P, D) tensor, got shape {tuple(t.shape)}")
    if t.shape[2] > 1 and t.stride(2) != 1:
        t = t.contiguous()
    return t


def ptr(t):
    return None if t is None else t.data_ptr()
