"""Ball query -- B200 drop-in for `pytorch3d.ops.ball_query`.

The call surface is pytorch3d's as recalled ([3P-memory]; parity with pytorch3d itself is unpinned).  Semantics
(include/pcl.h, "ball query"): for every query i < lengths1[n], the first K targets j < lengths2[n] in ascending index
order whose squared distance (the Chamfer / kNN arithmetic of `mode`, default cfg.chamfer_mode) is < radius * radius.
Empty slots and rows i >= lengths1[n] are dist 0, idx -1.  Gradients flow to both clouds through `dists` (and to p2
through `knn`); `idx` is not differentiable.

This is not pointnet2's `query_ball_point` (sampling.py): that one tests <= float32(radius ** 2) on xyz only, pads with
the first hit and has neither lengths, distances nor a gradient.
"""
import torch
from torch.autograd import Function

from . import _lib, cfg
from .chamfer import _MODES
from .knn import _KNN, _backward, _check_shapes, _lengths


def _check_k(K):
    if isinstance(K, bool) or int(K) != K or int(K) < 1:
        raise ValueError(f"K={K} must be a positive integer")


def _radius2(radius) -> float:
    """float32(radius) * float32(radius), rounded to fp32 (pytorch3d squares the radius inside its kernel)."""
    r = torch.tensor(float(radius), dtype=torch.float32)
    return float(r * r)


def ball_query_forward_raw(p1, p2, lengths1=None, lengths2=None, K=500, radius=0.2, mode=None):
    """One pcl_ball_query_fwd call.  Returns dict(dists (B,P1,K) fp32, idx (B,P1,K) int32, and the kernel's views of the
    inputs)."""
    _check_shapes(p1, p2, lengths1, lengths2)
    _check_k(K)
    K = int(K)
    _lib.require_cuda()
    L = _lib.lib()
    p1, p2 = _lib.as_points(p1), _lib.as_points(p2)
    if p2.device != p1.device:
        p2 = p2.to(p1.device)
    b, n1, d = p1.shape
    n2 = p2.shape[1]
    dev = p1.device
    mode = _MODES[cfg.chamfer_mode if mode is None else mode]
    l1, l2 = _lengths(lengths1, dev), _lengths(lengths2, dev)
    with _lib.on_device(dev):
        dists = torch.empty(b, n1, K, device=dev, dtype=torch.float32)
        idx = torch.empty(b, n1, K, device=dev, dtype=torch.int32)
        rc = L.pcl_ball_query_fwd(*_lib.pts_args(p1), _lib.ptr(l1), *_lib.pts_args(p2), _lib.ptr(l2), b, n1, n2, d, K,
                                  _radius2(radius), mode, dists.data_ptr(), idx.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_ball_query_fwd")
    return dict(dists=dists, idx=idx, p1=p1, p2=p2, len1=l1, len2=l2)


class _BallQueryFunction(Function):
    @staticmethod
    def forward(ctx, p1, p2, lengths1, lengths2, K, radius, mode):
        ctx.in_meta = (p1.dtype, p1.device, p2.dtype, p2.device)
        ctx.n_inputs = 7
        r = ball_query_forward_raw(p1, p2, lengths1, lengths2, K, radius, mode)
        ctx.save_for_backward(r["p1"], r["p2"], r["idx"])
        ctx.lens = (r["len1"], r["len2"])
        idx = r["idx"].long()
        ctx.mark_non_differentiable(idx)
        return r["dists"], idx

    @staticmethod
    def backward(ctx, grad_dists, grad_idx):
        return _backward(ctx, grad_dists, "pcl_ball_query_bwd")


def ball_query(p1, p2, lengths1=None, lengths2=None, K=500, radius=0.2, return_nn=True, *, mode=None):
    """Same call surface as pytorch3d.ops.ball_query [3P-memory].  Returns KNN(dists (N,P1,K) fp32, idx (N,P1,K) int64
    with -1 in empty slots, knn (N,P1,K,D) or None).  `knn` gathers p2 at idx and is zero in the empty slots
    (pytorch3d's masked_gather); it is plain torch indexing, so autograd reaches p2 through it too.

    The comparison value is float32(radius) * float32(radius) rounded to fp32, and the test is strict (<); pointnet2's
    `query_ball_point` compares <= float32(radius ** 2) instead."""
    _check_shapes(p1, p2, lengths1, lengths2)
    _check_k(K)
    dists, idx = _BallQueryFunction.apply(p1, p2, lengths1, lengths2, int(K), float(radius), mode)
    nn = None
    if return_nn:
        n, l, k = idx.shape
        u = p2.shape[2]
        keep = idx >= 0
        src = idx.clamp(min=0).to(p2.device)
        nn = p2.gather(1, src.reshape(n, l * k, 1).expand(-1, -1, u)).view(n, l, k, u)
        nn = torch.where(keep.to(p2.device)[..., None], nn, torch.zeros((), dtype=nn.dtype, device=nn.device))
    return _KNN(dists=dists, idx=idx, knn=nn)
