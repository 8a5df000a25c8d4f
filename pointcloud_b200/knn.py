"""K nearest neighbours -- B200 drop-in for `pytorch3d.ops.knn_points` / `knn_gather` with norm=2.

The call surface is pytorch3d's as recalled (SURVEY.md App. B style [3P-memory]; parity with pytorch3d itself is
unpinned).  Semantics (include/pcl.h, "k nearest neighbours"): squared L2 distances with the Chamfer arithmetic
(`mode`, default cfg.chamfer_mode), the K smallest targets of every query under the key (distance, index), sorted
ascending -- exact ties go to the lower index, NaN distances rank after +inf.  Slots k >= min(K, lengths2[n]) and rows
i >= lengths1[n] are 0.  Gradients flow to both clouds through `dists`; `idx` is not differentiable.
"""
from collections import namedtuple

import torch
from torch.autograd import Function

from . import _lib, cfg
from .chamfer import _MODES

_KNN = namedtuple("KNN", "dists idx knn")


def knn_max_k() -> int:
    return int(_lib.lib().pcl_knn_max_k())


def _check(p1, p2, K, lengths1=None, lengths2=None, norm=2):
    if norm != 2:
        raise NotImplementedError("only norm=2 (squared L2) is supported")
    _check_shapes(p1, p2, lengths1, lengths2)
    kmax = knn_max_k()
    if isinstance(K, bool) or int(K) != K or not 1 <= int(K) <= kmax:
        raise ValueError(f"K={K} is not supported (1..{kmax})")


def _check_shapes(p1, p2, lengths1=None, lengths2=None):
    """The shape checks shared by knn_points and ball_query (pytorch3d's messages)."""
    if p1.dim() != 3 or p2.dim() != 3:
        raise ValueError("Expected points to be of shape (N, P, D)")
    if p1.shape[0] != p2.shape[0]:
        raise ValueError("pts1 and pts2 must have the same batch dimension.")  # pytorch3d's message
    if p1.shape[2] != p2.shape[2]:
        raise ValueError("pts1 and pts2 must have the same point dimension.")  # pytorch3d's message
    if not 1 <= p1.shape[2] <= 8:
        raise ValueError(f"point dimension D={p1.shape[2]} is not supported (1..8)")
    for name, ln in (("lengths1", lengths1), ("lengths2", lengths2)):
        if ln is not None and ln.shape != (p1.shape[0],):
            raise ValueError(f"Expected {name} to be of shape (N,).")


def _lengths(lengths, dev):
    if lengths is None:
        return None
    return lengths.to(device=dev, dtype=torch.int64).contiguous()


def knn_forward_raw(p1, p2, lengths1=None, lengths2=None, K=1, mode=None):
    """One pcl_knn_fwd call.  Returns dict(dists (B,P1,K) fp32, idx (B,P1,K) int32, and the kernel's views of the inputs)."""
    K = int(K)
    _check(p1, p2, K, lengths1, lengths2)
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
        rc = L.pcl_knn_fwd(*_lib.pts_args(p1), _lib.ptr(l1), *_lib.pts_args(p2), _lib.ptr(l2), b, n1, n2, d, K, mode,
                           dists.data_ptr(), idx.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_knn_fwd")
    return dict(dists=dists, idx=idx, p1=p1, p2=p2, len1=l1, len2=l2)


class _KnnFunction(Function):
    @staticmethod
    def forward(ctx, p1, p2, lengths1, lengths2, K, mode):
        ctx.in_meta = (p1.dtype, p1.device, p2.dtype, p2.device)
        ctx.n_inputs = 6
        r = knn_forward_raw(p1, p2, lengths1, lengths2, K, mode)
        ctx.save_for_backward(r["p1"], r["p2"], r["idx"])
        ctx.lens = (r["len1"], r["len2"])
        idx = r["idx"].long()
        ctx.mark_non_differentiable(idx)
        return r["dists"], idx

    @staticmethod
    def backward(ctx, grad_dists, grad_idx):
        return _backward(ctx, grad_dists, "pcl_knn_bwd")


def _backward(ctx, grad_dists, entry):
    """Gradients of (p1, p2) through dists with `entry` (pcl_knn_bwd or pcl_ball_query_bwd), cast back to the inputs'
    dtypes and devices; None for the other forward arguments."""
    p1, p2, idx = ctx.saved_tensors
    l1, l2 = ctx.lens
    L = _lib.lib()
    b, n1, d = p1.shape
    n2, K = p2.shape[1], idx.shape[2]
    dev = p1.device
    g = grad_dists.to(device=dev, dtype=torch.float32).contiguous()  # read on the device: no host sync
    with _lib.on_device(dev):
        g1 = torch.empty(b, n1, d, device=dev, dtype=torch.float32)
        g2 = torch.empty(b, n2, d, device=dev, dtype=torch.float32)
        rc = getattr(L, entry)(*_lib.pts_args(p1), _lib.ptr(l1), *_lib.pts_args(p2), _lib.ptr(l2), b, n1, n2, d, K,
                               idx.data_ptr(), g.data_ptr(), g1.data_ptr(), g2.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, entry)
    dt1, dev1, dt2, dev2 = ctx.in_meta
    return (g1.to(device=dev1, dtype=dt1), g2.to(device=dev2, dtype=dt2)) + (None,) * (ctx.n_inputs - 2)


def knn_gather(x, idx, lengths=None):
    """pytorch3d.ops.knn_gather: x (N, M, U), idx (N, L, K) -> (N, L, K, U) = x[n, idx[n, l, k]]; slots k >= lengths[n]
    are zero.  Plain torch indexing (autograd gives the backward); no host synchronisation."""
    n, _, u = x.shape
    n2, l, k = idx.shape
    if n != n2:
        raise ValueError("x and idx must have same batch dimension.")  # pytorch3d's message
    idx = idx.to(x.device).long()
    out = x.gather(1, idx.reshape(n, l * k, 1).expand(-1, -1, u)).view(n, l, k, u)
    if lengths is not None:
        keep = torch.arange(k, device=x.device)[None, :] < lengths.to(x.device).view(n, 1)
        out = torch.where(keep[:, None, :, None], out, torch.zeros((), dtype=out.dtype, device=out.device))
    return out


def knn_points(p1, p2, lengths1=None, lengths2=None, norm=2, K=1, version=-1, return_nn=False, return_sorted=True, *,
               mode=None):
    """Same call surface as pytorch3d.ops.knn_points [3P-memory].  Returns KNN(dists (N,P1,K) fp32, idx (N,P1,K) int64,
    knn (N,P1,K,D) or None).  Results are always sorted (pytorch3d leaves the order unspecified for return_sorted=False);
    `version` selects a pytorch3d kernel variant and is ignored."""
    _check(p1, p2, K, lengths1, lengths2, norm)
    dists, idx = _KnnFunction.apply(p1, p2, lengths1, lengths2, int(K), mode)
    nn = knn_gather(p2, idx, lengths2) if return_nn else None
    return _KNN(dists=dists, idx=idx, knn=nn)
