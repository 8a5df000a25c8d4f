"""Point compositors -- B200 drop-ins for `pytorch3d.renderer.compositing`'s alpha_composite, norm_weighted_sum and
weighted_sum.

The semantics are pytorch3d 0.7.2's as recalled ([3P-memory]; parity with pytorch3d itself is unpinned): tests/raster_ref.py
restates them in torch and is the specification.  pointsidx (N, K, H, W) int32 / int64 indexes the columns of
pt_clds (C, P_total); alphas (N, K, H, W).  The output is (N, C, H, W) fp32, summed in fp32 in k order:
  weighted_sum:       sum_k a_k F[:, idx_k]
  norm_weighted_sum:  sum_k (a_k F[:, idx_k]) / w,  w = max(sum of the valid a_k, 1e-4)
  alpha_composite:    sum_k ((T_k a_k) F[:, idx_k]),  T_k = prod_{t<k} (1 - a_t) over every t < k, valid or not.
A slot with idx < 0 or idx >= P_total contributes nothing.  All three inputs are read through their strides, so the
renderer's `idx.permute(0, 3, 1, 2)` and `features_packed().t()` need no copy.  Gradients are the exact derivatives
(alpha_composite's from products of (1 - a_t), so a = 1 stays finite); they come back in each input's dtype and on its
device; pointsidx gets none.
"""
import ctypes

import torch
from torch.autograd import Function

from . import _lib

ALPHA, NORM_WEIGHTED, WEIGHTED = 0, 1, 2


def _strides(t):
    return (ctypes.c_int64 * t.dim())(*t.stride())


def _inputs(pointsidx, alphas, pt_clds):
    if pointsidx.dim() != 4 or alphas.dim() != 4 or tuple(alphas.shape) != tuple(pointsidx.shape):
        raise ValueError(f"pointsidx and alphas must both be (N, K, H, W), got {tuple(pointsidx.shape)} and "
                         f"{tuple(alphas.shape)}")
    if pt_clds.dim() != 2:
        raise ValueError(f"pt_clds must be (C, P), got {tuple(pt_clds.shape)}")
    if pointsidx.dtype not in (torch.int32, torch.int64):
        raise ValueError(f"pointsidx must be int32 or int64, got {pointsidx.dtype}")
    if not alphas.is_cuda:
        _lib.require_cuda()
    dev = alphas.device if alphas.is_cuda else torch.device("cuda")
    idx = pointsidx.to(dev)
    a = alphas.to(device=dev, dtype=torch.float32)
    f = pt_clds.to(device=dev, dtype=torch.float32)
    return idx, a, f


def _args(mode, idx, a, f):
    n, k, h, w = idx.shape
    return [mode, idx.data_ptr(), int(idx.dtype == torch.int64), _strides(idx), a.data_ptr(), _strides(a), f.data_ptr(),
            _strides(f), n, k, h, w, f.shape[0], f.shape[1]]


def composite_forward_raw(mode, pointsidx, alphas, pt_clds):
    """pcl_composite_fwd: one C call, no autograd.  -> (N, C, H, W) fp32."""
    idx, a, f = _inputs(pointsidx, alphas, pt_clds)
    dev = a.device
    n, _, h, w = idx.shape
    with _lib.on_device(dev):
        out = torch.empty(n, f.shape[0], h, w, device=dev, dtype=torch.float32)
        rc = _lib.lib().pcl_composite_fwd(*_args(mode, idx, a, f), out.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_composite_fwd")
    return out


class _CompositeFunction(Function):
    @staticmethod
    def forward(ctx, mode, pointsidx, alphas, pt_clds):
        ctx.set_materialize_grads(False)
        idx, a, f = _inputs(pointsidx, alphas, pt_clds)
        out = composite_forward_raw(mode, idx, a, f)
        ctx.save_for_backward(idx, a, f)
        ctx.mode = mode
        ctx.meta = (alphas.dtype, alphas.device, pt_clds.dtype, pt_clds.device)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        idx, a, f = ctx.saved_tensors
        want_a, want_f = ctx.needs_input_grad[2], ctx.needs_input_grad[3]
        if grad_out is None or not (want_a or want_f):
            return None, None, None, None
        dev = a.device
        g = grad_out.to(device=dev, dtype=torch.float32).contiguous()
        with _lib.on_device(dev):
            ga = torch.empty(a.shape, device=dev, dtype=torch.float32) if want_a else None
            gf = torch.empty(f.shape, device=dev, dtype=torch.float32) if want_f else None
            rc = _lib.lib().pcl_composite_bwd(*_args(ctx.mode, idx, a, f), g.data_ptr(), _lib.ptr(ga), _lib.ptr(gf),
                                              _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_composite_bwd")
        adt, adev, fdt, fdev = ctx.meta
        ga = None if ga is None else ga.to(device=adev, dtype=adt)
        gf = None if gf is None else gf.to(device=fdev, dtype=fdt)
        return None, None, ga, gf


def alpha_composite(pointsidx, alphas, pt_clds):
    """pytorch3d.renderer.compositing.alpha_composite [3P-memory]: front-to-back alpha compositing of the K points of every
    pixel.  pointsidx (N, K, H, W) int32 / int64, alphas (N, K, H, W), pt_clds (C, P) -> (N, C, H, W) fp32."""
    return _CompositeFunction.apply(ALPHA, pointsidx, alphas, pt_clds)


def norm_weighted_sum(pointsidx, alphas, pt_clds):
    """pytorch3d.renderer.compositing.norm_weighted_sum [3P-memory]: the alpha-weighted mean of the pixel's point features
    (weights summed over the valid slots, clamped below at 1e-4).  Shapes as alpha_composite."""
    return _CompositeFunction.apply(NORM_WEIGHTED, pointsidx, alphas, pt_clds)


def weighted_sum(pointsidx, alphas, pt_clds):
    """pytorch3d.renderer.compositing.weighted_sum [3P-memory]: the alpha-weighted sum of the pixel's point features.
    Shapes as alpha_composite."""
    return _CompositeFunction.apply(WEIGHTED, pointsidx, alphas, pt_clds)
