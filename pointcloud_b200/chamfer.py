"""Chamfer distance -- B200 drop-in for `pytorch3d.loss.chamfer_distance` (0.7.2).  The reference calls
`chamfer_distance(pred, target)[0]` (pointcloud_vision/utils.py:211) and `chamfer_distance(pred, target, y_lengths=...)[0]`
(:228); normals, weights and batch_reduction None / "sum" are the rest of pytorch3d's call surface.

Semantics restated from pytorch3d 0.7.2 (SURVEY.md App. B; parity unpinned -- pytorch3d is not available):
squared-L2 K=1 nearest neighbour in both directions (lowest index on exact ties), padded points ignored,
point_reduction="mean", loss = cham_x + cham_y; both clouds receive gradient.  The default call (no normals pair, no weights,
batch_reduction="mean") runs pcl_chamfer_fwd / pcl_chamfer_bwd; every other call runs pcl_chamfer_cloud_fwd / _bwd, which also
return per-cloud sums and the normal term, and composes the (N,)-sized reductions in torch.
"""
import torch
from torch.autograd import Function

from . import _lib, cfg

_MODES = {"unfused": _lib.PCL_CHAMFER_UNFUSED, "fma": _lib.PCL_CHAMFER_FMA, 0: 0, 1: 1}


def _lengths(lengths, b, p, dev, name):
    if lengths is None:
        return None
    if lengths.shape != (b,):
        raise ValueError(f"Expected {name} to be of shape (N,).")  # pytorch3d's message
    return lengths.to(device=dev, dtype=torch.int64).contiguous()


def _normals(nrm, b, p, dev, name):
    if nrm is None:
        return None
    if nrm.dim() != 3 or tuple(nrm.shape) != (b, p, 3):
        raise ValueError(f"Expected {name} to be of shape (N, P, 3).")
    nrm = _lib.as_points(nrm)
    return nrm if nrm.device == dev else nrm.to(dev)


_NO_PTS = [None, _lib.PCL_F32, 0, 0]


def chamfer_forward_raw(x, y, x_lengths=None, y_lengths=None, mode=None, *, x_normals=None, y_normals=None, cloud_sums=False):
    """One pcl_chamfer_fwd call.  Returns dict(loss_xy (2,) batch means, loss_sums (2,) batch sums, dist_x, idx_x, dist_y, idx_y).
    With cloud_sums=True, or with both x_normals and y_normals ((N, P, 3), any float dtype, strided views read in place), it is
    one pcl_chamfer_cloud_fwd call instead, which also returns cloud_sums (2, N): every cloud's un-normalised sum of distances
    per direction, and normal_sums (2, N): every cloud's sum of 1 - |cos| over its points (None without both normals)."""
    _lib.require_cuda()
    L = _lib.lib()
    x, y = _lib.as_points(x), _lib.as_points(y)
    if y.device != x.device:
        y = y.to(x.device)
    b, p1, d = x.shape
    if y.shape[0] != b or y.shape[2] != d:
        raise ValueError("y does not have the correct shape.")  # pytorch3d's message
    p2 = y.shape[1]
    dev = x.device
    mode = _MODES[cfg.chamfer_mode if mode is None else mode]
    xl, yl = _lengths(x_lengths, b, p1, dev, "x_lengths"), _lengths(y_lengths, b, p2, dev, "y_lengths")
    xn, yn = _normals(x_normals, b, p1, dev, "normals"), _normals(y_normals, b, p2, dev, "normals")
    if xn is None or yn is None:
        xn = yn = None
    cloud = cloud_sums or xn is not None
    with _lib.on_device(dev):
        dist_x = torch.empty(b, p1, device=dev, dtype=torch.float32); idx_x = torch.empty(b, p1, device=dev, dtype=torch.int32)
        dist_y = torch.empty(b, p2, device=dev, dtype=torch.float32); idx_y = torch.empty(b, p2, device=dev, dtype=torch.int32)
        loss4 = torch.empty(4, device=dev, dtype=torch.float32)
        wsb = L.pcl_chamfer_workspace_bytes(b, p1, p2)
        ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
        if not cloud:
            rc = L.pcl_chamfer_fwd(*_lib.pts_args(x), _lib.ptr(xl), *_lib.pts_args(y), _lib.ptr(yl), b, p1, p2, d, mode,
                                   dist_x.data_ptr(), idx_x.data_ptr(), dist_y.data_ptr(), idx_y.data_ptr(),
                                   loss4.data_ptr(), ws.data_ptr(), wsb, _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_chamfer_fwd")
            return dict(loss_xy=loss4[:2], loss_sums=loss4[2:], dist_x=dist_x, idx_x=idx_x, dist_y=dist_y, idx_y=idx_y, x=x, y=y,
                        x_len=xl, y_len=yl)
        sums = torch.empty(2, b, device=dev, dtype=torch.float32)
        nsums = torch.empty(2, b, device=dev, dtype=torch.float32) if xn is not None else None
        nargs = _lib.pts_args(xn) + _lib.pts_args(yn) if xn is not None else _NO_PTS + _NO_PTS
        rc = L.pcl_chamfer_cloud_fwd(*_lib.pts_args(x), _lib.ptr(xl), *_lib.pts_args(y), _lib.ptr(yl), b, p1, p2, d, mode,
                                     dist_x.data_ptr(), idx_x.data_ptr(), dist_y.data_ptr(), idx_y.data_ptr(), loss4.data_ptr(),
                                     sums.data_ptr(), *nargs, _lib.ptr(nsums), ws.data_ptr(), wsb, _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_chamfer_cloud_fwd")
    return dict(loss_xy=loss4[:2], loss_sums=loss4[2:], dist_x=dist_x, idx_x=idx_x, dist_y=dist_y, idx_y=idx_y, x=x, y=y,
                x_len=xl, y_len=yl, cloud_sums=sums, normal_sums=nsums, x_normals=xn, y_normals=yn)


class _ChamferFunction(Function):
    @staticmethod
    def forward(ctx, x, y, x_lengths, y_lengths, mode):
        ctx.in_meta = (x.dtype, x.device, y.dtype, y.device)
        r = chamfer_forward_raw(x, y, x_lengths, y_lengths, mode)
        ctx.save_for_backward(r["x"], r["y"], r["idx_x"], r["idx_y"])
        ctx.lens = (r["x_len"], r["y_len"])
        return r["loss_xy"]

    @staticmethod
    def backward(ctx, grad_xy):
        x, y, idx_x, idx_y = ctx.saved_tensors
        xl, yl = ctx.lens
        L = _lib.lib()
        b, p1, d = x.shape
        p2 = y.shape[1]
        dev = x.device
        grad_xy = grad_xy.contiguous().float()
        with _lib.on_device(dev):
            gx = torch.empty(b, p1, d, device=dev, dtype=torch.float32)
            gy = torch.empty(b, p2, d, device=dev, dtype=torch.float32)
            g = grad_xy  # (2,): upstream gradients of loss_x and loss_y, read on the device
            rc = L.pcl_chamfer_bwd(*_lib.pts_args(x), _lib.ptr(xl), *_lib.pts_args(y), _lib.ptr(yl), b, p1, p2, d,
                                   idx_x.data_ptr(), idx_y.data_ptr(), g.data_ptr(), gx.data_ptr(), gy.data_ptr(),
                                   _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_chamfer_bwd")
        dtx, devx, dty, devy = ctx.in_meta
        return gx.to(device=devx, dtype=dtx), gy.to(device=devy, dtype=dty), None, None, None


def _clamped_lengths(lengths, b, p, dev):
    """clamp(len, 1) as float32 (N,): the point-mean denominators."""
    if lengths is None:
        return torch.full((b,), float(max(p, 1)), device=dev, dtype=torch.float32)
    return lengths.clamp(min=1).to(torch.float32)


class _ChamferCloudFunction(Function):
    """pcl_chamfer_cloud_fwd / pcl_chamfer_cloud_bwd: returns loss_xy (2,) (the batch means, as _ChamferFunction), cloud_sums
    (2, N) and normal_sums (2, N) (None without both normals); the backward takes the upstream gradients of all three."""

    @staticmethod
    def forward(ctx, x, y, x_lengths, y_lengths, x_normals, y_normals, mode):
        ctx.in_meta = (x.dtype, x.device, y.dtype, y.device)
        ctx.nrm_meta = None if x_normals is None else (x_normals.dtype, x_normals.device, y_normals.dtype, y_normals.device)
        r = chamfer_forward_raw(x, y, x_lengths, y_lengths, mode, x_normals=x_normals, y_normals=y_normals, cloud_sums=True)
        ctx.save_for_backward(r["x"], r["y"], r["idx_x"], r["idx_y"], r["x_normals"], r["y_normals"])
        ctx.lens = (r["x_len"], r["y_len"])
        return r["loss_xy"], r["cloud_sums"], r["normal_sums"]

    @staticmethod
    def backward(ctx, grad_xy, grad_cloud, grad_normal):
        x, y, idx_x, idx_y, xn, yn = ctx.saved_tensors
        xl, yl = ctx.lens
        L = _lib.lib()
        b, p1, d = x.shape
        p2 = y.shape[1]
        dev = x.device
        with _lib.on_device(dev):
            # loss_xy[d] = sum_n cloud_sums[d, n] / clamp(len, 1) / max(N, 1): its gradient joins the per-cloud one with
            # pcl_chamfer_bwd's arithmetic (g / B / len, true divisions)
            den = torch.stack([_clamped_lengths(xl, b, p1, dev), _clamped_lengths(yl, b, p2, dev)])
            nb = torch.full((1, 1), float(max(b, 1)), device=dev, dtype=torch.float32)
            gc = (grad_xy.float()[:, None] / nb / den + grad_cloud.float()).contiguous()
            gx = torch.empty(b, p1, d, device=dev, dtype=torch.float32)
            gy = torch.empty(b, p2, d, device=dev, dtype=torch.float32)
            gxn = gyn = gn = None
            if xn is not None and grad_normal is not None:
                gn = grad_normal.float().contiguous()
                gxn = torch.empty(b, p1, 3, device=dev, dtype=torch.float32)
                gyn = torch.empty(b, p2, 3, device=dev, dtype=torch.float32)
            nargs = _lib.pts_args(xn) + _lib.pts_args(yn) if gn is not None else _NO_PTS + _NO_PTS
            rc = L.pcl_chamfer_cloud_bwd(*_lib.pts_args(x), _lib.ptr(xl), *_lib.pts_args(y), _lib.ptr(yl), b, p1, p2, d,
                                         idx_x.data_ptr(), idx_y.data_ptr(), gc.data_ptr(), gx.data_ptr(), gy.data_ptr(), *nargs,
                                         _lib.ptr(gn), _lib.ptr(gxn), _lib.ptr(gyn), _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_chamfer_cloud_bwd")
        dtx, devx, dty, devy = ctx.in_meta
        if gxn is not None:
            ndx, ndevx, ndy, ndevy = ctx.nrm_meta
            gxn, gyn = gxn.to(device=ndevx, dtype=ndx), gyn.to(device=ndevy, dtype=ndy)
        return gx.to(device=devx, dtype=dtx), gy.to(device=devy, dtype=dty), None, None, gxn, gyn, None


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None, weights=None,
                     batch_reduction="mean", point_reduction="mean", norm=2, *, mode=None):
    """pytorch3d.loss.chamfer_distance (0.7.2): returns (loss, loss_normals).

    loss: per cloud, the point mean of the squared distance to the nearest neighbour, in both directions, summed
    (cham_x + cham_y); times weights[n] when weights are given; batch_reduction None returns it per cloud (N,), "sum" sums
    over the clouds and "mean" divides that sum by weights.sum() (or by max(N, 1) without weights).
    loss_normals: computed only when both x_normals and y_normals ((N, P, 3)) are given, else None: 1 - |cos| between each
    point's normal and its nearest neighbour's (F.cosine_similarity, eps=1e-6), with the same weights and reductions; a point
    whose target cloud is empty adds 1.  Points get the gradient of loss only; both normals get that of loss_normals.
    point_reduction="sum" and norm=1 raise NotImplementedError.

    Host synchronisation: with weights, the checks that no weight is negative and whether all are zero read the weights on
    the host, as pytorch3d does; all-zero weights return zeros that stay attached to the graph.  Without weights no call
    here synchronises with the host.
    """
    if point_reduction != "mean" or norm != 2:
        raise NotImplementedError("only point_reduction='mean' and norm=2 (squared L2, pytorch3d's defaults)")
    if batch_reduction is not None and batch_reduction not in ("mean", "sum"):
        raise ValueError('batch_reduction must be one of ["mean", "sum"] or None')  # pytorch3d's message
    if x.dim() != 3 or y.dim() != 3:
        raise ValueError("Expected points to be of shape (N, P, D)")
    n = x.shape[0]
    for nrm, pts in ((x_normals, x), (y_normals, y)):
        if nrm is not None and (nrm.dim() != 3 or tuple(nrm.shape) != (n, pts.shape[1], 3)):
            raise ValueError("Expected normals to be of shape (N, P, 3)")
    both_normals = x_normals is not None and y_normals is not None
    if weights is not None:
        if weights.dim() != 1 or weights.size(0) != n:
            raise ValueError("weights must be of shape (N,).")  # pytorch3d's messages
        if not (weights >= 0).all():
            raise ValueError("weights cannot be negative.")
        if weights.sum() == 0.0:
            def zero():
                z = x.sum((1, 2)) * weights.to(x.device) * 0.0
                return z.sum() if batch_reduction is not None else z
            return zero(), zero()
    if weights is None and batch_reduction == "mean" and not both_normals:
        loss_xy = _ChamferFunction.apply(x, y, x_lengths, y_lengths, mode)
        return loss_xy[0] + loss_xy[1], None
    loss_xy, sums, nsums = _ChamferCloudFunction.apply(x, y, x_lengths, y_lengths, x_normals if both_normals else None,
                                                       y_normals if both_normals else None, mode)
    dev = sums.device
    den = torch.stack([_clamped_lengths(None if x_lengths is None else x_lengths.to(dev), n, x.shape[1], dev),
                       _clamped_lengths(None if y_lengths is None else y_lengths.to(dev), n, y.shape[1], dev)])
    w = None if weights is None else weights.to(dev)

    def reduce(s):  # (2, N) per-cloud sums -> the loss
        per = s / den
        if w is not None:
            per = per * w
        if batch_reduction is None:
            return per[0] + per[1]
        cx, cy = per[0].sum(), per[1].sum()
        if batch_reduction == "mean":
            div = w.sum() if w is not None else max(n, 1)
            cx, cy = cx / div, cy / div
        return cx + cy

    if weights is None and batch_reduction == "mean":
        loss = loss_xy[0] + loss_xy[1]  # the same scalar as the call without normals, bit for bit
    else:
        loss = reduce(sums)
    return loss, (reduce(nsums) if nsums is not None else None)
