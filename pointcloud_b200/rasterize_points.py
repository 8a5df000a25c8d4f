"""Rasterize points -- B200 drop-in for `pytorch3d.renderer.points.rasterize_points`.

The semantics are pytorch3d 0.7.2's as recalled ([3P-memory]; parity with pytorch3d itself is unpinned): tests/raster_ref.py
restates them in torch and is the specification; include/pcl.h ("rasterize points / compositing") says the same in C terms.
points (B, P, 3) are in NDC (+X left, +Y up, +Z away from the camera); cloud b is points[b, :lengths[b]] (lengths clamped to
[0, P]).  Pixel (row r, column c) of the H x W image has the fp32 centre (ndc(W-1-c, W, H), ndc(H-1-r, H, W)) with
ndc(i, S1, S2) = -off + (range*i + off) / S1, range = S1 > S2 ? (S1*2)/S2 : 2, off = range/2, so the shorter side spans
[-1, 1].  A point hits the pixel when its x, y, z and radius are finite, z >= 0 and d2 = dx*dx + dy*dy <= r*r (fp32, every
operation rounded).  The pixel keeps the K hits of smallest (z, index), z = -0.0 counting as +0.0, ascending:
idx (B, H, W, K) int32 holds the packed index sum(lengths[:b]) + i, zbuf the point's z, dists d2; unused slots are -1.

Differences from pytorch3d, deliberate:
  - a non-finite coordinate or radius never hits (pytorch3d's skips let NaN through);
  - every operation is rounded (pytorch3d's nvcc build may contract into FMAs);
  - ties in z are broken by index;
  - bin_size=None picks 0 for clouds of up to 4096 points and 16 above;
  - bins that overflow `max_points_per_bin` are rasterized from the whole cloud instead of raising, so nothing is read
    back to the host; `bin_size` must be 0 or a multiple of 16;
  - ragged clouds come as `lengths=` instead of a `Pointclouds` object.

Gradients: zbuf's slot adds its gradient to the point's z, dists' slot adds 2 * g * (p_xy - pixel_xy) to its x and y;
-1 slots and points that land in no slot give exactly 0.  radius and lengths get none.  They come back in the points'
dtype and on their device.
"""
import torch
from torch.autograd import Function

from . import _lib

MAX_POINTS_PER_PIXEL = 150


def _image_size(image_size):
    if isinstance(image_size, int):
        return image_size, image_size
    h, w = (int(s) for s in image_size)
    return h, w


def _check(points, lengths, image_size, radius, points_per_pixel, bin_size, max_points_per_bin):
    """pytorch3d's ValueErrors, plus the limits of the kernels.  Reads nothing from the device."""
    if points.dim() != 3 or points.shape[2] != 3:
        raise ValueError(f"points must be of shape (N, P, 3), got {tuple(points.shape)}")
    b, p, _ = points.shape
    if points_per_pixel > MAX_POINTS_PER_PIXEL:
        raise ValueError(f"Must have points_per_pixel <= {MAX_POINTS_PER_PIXEL}")
    if points_per_pixel < 1:
        raise ValueError("points_per_pixel must be at least 1")
    h, w = _image_size(image_size)
    if not (1 <= h <= 16384 and 1 <= w <= 16384):
        raise ValueError(f"image_size {(h, w)}: each side must be in 1..16384")
    if torch.is_tensor(radius) and tuple(radius.shape) != (b, p):
        raise ValueError("radius must be a float or a tensor of shape (N, P)")
    if lengths is not None and tuple(lengths.shape) != (b,):
        raise ValueError(f"lengths must be of shape (N,), got {tuple(lengths.shape)}")
    if bin_size is not None and (bin_size < 0 or bin_size % 16):
        raise ValueError(f"bin_size={bin_size} must be None, 0 or a positive multiple of 16")
    if b * p >= 2 ** 31:
        raise ValueError("N * P must be below 2^31")
    return h, w


def auto_bin_size(P):
    """bin_size=None.  Of 0 (no bins), 16, 32, 64 and 128, bins of 16 x 16 pixels were the fastest from P = 16384 up on
    every shape of tools/rasterize_points_time.py.  At P = 2048 (B=32, 128 x 128) their edge over no bins was small and
    did not hold forward+backward in every run of the tool, so clouds of up to 4096 points take no bins and are never
    slower than bin_size=0 (DESIGN.md section 3.4)."""
    return 0 if P <= 4096 else 16


def rasterize_points_forward_raw(points, lengths=None, image_size=256, radius=0.01, points_per_pixel=8, bin_size=None,
                                 max_points_per_bin=None):
    """pcl_rasterize_points_fwd: one C call, no autograd, capturable in a CUDA graph.  Returns dict(idx (B,H,W,K) int32,
    zbuf, dists (B,H,W,K) fp32, and the kernels' views: points, lengths (int64 or None), radius (fp32 (B,P) or None))."""
    h, w = _check(points, lengths, image_size, radius, points_per_pixel, bin_size, max_points_per_bin)
    p = _lib.as_points(points)
    dev = p.device
    b, n, _ = p.shape
    ln = None if lengths is None else lengths.to(device=dev, dtype=torch.int64).contiguous()
    rad = radius.to(device=dev, dtype=torch.float32).contiguous() if torch.is_tensor(radius) else None
    rs = 0.0 if rad is not None else float(radius)
    bs = auto_bin_size(n) if bin_size is None else int(bin_size)
    mppb = 0 if max_points_per_bin is None else int(max_points_per_bin)
    K = int(points_per_pixel)
    L = _lib.lib()
    with _lib.on_device(dev):
        idx = torch.empty(b, h, w, K, device=dev, dtype=torch.int32)
        zbuf = torch.empty(b, h, w, K, device=dev, dtype=torch.float32)
        dists = torch.empty(b, h, w, K, device=dev, dtype=torch.float32)
        nws = int(L.pcl_rasterize_points_workspace_bytes(b, n, h, w, bs, mppb))
        ws = torch.empty(max(nws, 1), device=dev, dtype=torch.uint8)
        rc = L.pcl_rasterize_points_fwd(*_lib.pts_args(p), _lib.ptr(ln), _lib.ptr(rad), rs, b, n, h, w, K, bs, mppb,
                                        idx.data_ptr(), zbuf.data_ptr(), dists.data_ptr(), ws.data_ptr(), nws,
                                        _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_rasterize_points_fwd")
    return dict(idx=idx, zbuf=zbuf, dists=dists, points=p, lengths=ln, radius=rad)


def rasterize_points_backward_raw(points, lengths, idx, grad_zbuf, grad_dists):
    """pcl_rasterize_points_bwd: -> grad_points (B, P, 3) fp32 on the points' device (the kernels' view of `points`)."""
    p = _lib.as_points(points)
    dev = p.device
    b, n, _ = p.shape
    _, h, w, K = idx.shape
    ln = None if lengths is None else lengths.to(device=dev, dtype=torch.int64).contiguous()

    def f32(g):
        return None if g is None else g.to(device=dev, dtype=torch.float32).contiguous()
    gz, gd = f32(grad_zbuf), f32(grad_dists)
    with _lib.on_device(dev):
        gp = torch.empty(b, n, 3, device=dev, dtype=torch.float32)
        rc = _lib.lib().pcl_rasterize_points_bwd(*_lib.pts_args(p), _lib.ptr(ln), b, n, h, w, K, idx.contiguous().data_ptr(),
                                                 _lib.ptr(gz), _lib.ptr(gd), gp.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_rasterize_points_bwd")
    return gp


class _RasterizePointsFunction(Function):
    @staticmethod
    def forward(ctx, points, lengths, image_size, radius, points_per_pixel, bin_size, max_points_per_bin):
        ctx.set_materialize_grads(False)
        r = rasterize_points_forward_raw(points, lengths, image_size, radius, points_per_pixel, bin_size, max_points_per_bin)
        ctx.save_for_backward(points, r["lengths"], r["idx"])
        ctx.mark_non_differentiable(r["idx"])
        return r["idx"], r["zbuf"], r["dists"]

    @staticmethod
    def backward(ctx, grad_idx, grad_zbuf, grad_dists):
        points, lengths, idx = ctx.saved_tensors
        if not ctx.needs_input_grad[0] or (grad_zbuf is None and grad_dists is None):
            return None, None, None, None, None, None, None
        gp = rasterize_points_backward_raw(points, lengths, idx, grad_zbuf, grad_dists)
        return gp.to(device=points.device, dtype=points.dtype), None, None, None, None, None, None


def rasterize_points(points, lengths=None, image_size=256, radius=0.01, points_per_pixel=8, bin_size=None,
                     max_points_per_bin=None):
    """pytorch3d.renderer.points.rasterize_points [3P-memory] for padded clouds.

    points (N, P, 3) in NDC, fp32 / fp16 / bf16 read in place (strided views included; other floating types go through
    `.float()`); lengths (N,) int or None (every row counts); image_size an int or (H, W); radius a float or an (N, P)
    tensor; points_per_pixel K in 1..150; bin_size None (automatic), 0 (no bins) or a multiple of 16; max_points_per_bin
    None (max(10000, P/5)) or the capacity of a bin.  Returns (idx (N,H,W,K) int32, zbuf (N,H,W,K), dists (N,H,W,K)),
    differentiable in the points through zbuf and dists; see the module docstring.  The outputs do not depend on bin_size
    or max_points_per_bin.  Nothing on the path reads device data on the host."""
    _check(points, lengths, image_size, radius, points_per_pixel, bin_size, max_points_per_bin)
    return _RasterizePointsFunction.apply(points, lengths, image_size, radius, points_per_pixel, bin_size,
                                          max_points_per_bin)
