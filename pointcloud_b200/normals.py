"""Normals and local coordinate frames -- B200 drop-in for `pytorch3d.ops.estimate_pointcloud_normals` /
`estimate_pointcloud_local_coord_frames`.

The call surface is pytorch3d 0.7.2's as recalled ([3P-memory]; parity with pytorch3d itself is unpinned).  Semantics
(include/pcl.h, "normals and local frames"): the K neighbours of every point are `knn_points(p, p, lengths, lengths, K)`
(the point itself included); the mean and covariance of those K points are eigen-decomposed, eigenvalues ascending
(`curvatures`) and eigenvector c in column c of `frames`; with `disambiguate_directions` the first and last vectors are
oriented so that at least half of the neighbours project non-negatively on them, and the middle column is their cross
product.  `normals` is column 0.

Differences from pytorch3d: the per-point arithmetic is fp64 and rounded to fp32 once (pytorch3d works in fp32 and first
subtracts each cloud's mean, which only fp32 needs); ragged batches take `lengths=` instead of a `Pointclouds` object;
`use_symeig_workaround` is accepted and ignored (there is one solver); rows past a cloud's length are 0.  Neighbourhoods
with repeated eigenvalues (K = 1, duplicate or collinear points) get a finite orthonormal frame, but their gradient is
non-finite, as with torch.linalg.eigh.  Gradients reach the points through curvatures, frames and normals; they come
back in the points' dtype and on their device.
"""
import torch
from torch.autograd import Function

from . import _lib
from .knn import knn_forward_raw, knn_max_k

_SHAPE_MSG = "The pointclouds argument has to be of shape (minibatch, N, 3)"  # pytorch3d's messages
_SIZE_MSG = "The neighborhood_size argument has to be >= size of each of the point clouds."


def _check(points, K, lengths):
    """pytorch3d's checks plus 1 <= K <= knn_max_k().  With lengths, the size check reads them on the host."""
    if points.dim() != 3 or points.shape[2] != 3:
        raise ValueError(_SHAPE_MSG)
    kmax = knn_max_k()
    if isinstance(K, bool) or int(K) != K or not 1 <= int(K) <= kmax:
        raise ValueError(f"neighborhood_size={K} is not supported (1..{kmax})")
    K = int(K)
    b, p = points.shape[:2]
    if lengths is not None:
        if lengths.shape != (b,):
            raise ValueError("Expected lengths to be of shape (N,).")
        if b > 0 and bool((lengths.clamp(max=p) <= K).any()):
            raise ValueError(_SIZE_MSG)
    elif b > 0 and p <= K:
        raise ValueError(_SIZE_MSG)
    return K


def frames_forward_raw(points, neighborhood_size=50, disambiguate_directions=True, lengths=None, mode=None):
    """pcl_knn_fwd + pcl_frames_fwd.  Returns dict(curvatures (B,P,3) fp32, frames (B,P,3,3) fp32, idx (B,P,K) int32 -- the
    neighbours used, points -- the kernels' view of the input, lengths)."""
    K = _check(points, neighborhood_size, lengths)
    r = knn_forward_raw(points, points, lengths, lengths, K, mode)
    p, ln, idx = r["p1"], r["len1"], r["idx"]
    b, n, _ = p.shape
    dev = p.device
    L = _lib.lib()
    with _lib.on_device(dev):
        curv = torch.empty(b, n, 3, device=dev, dtype=torch.float32)
        frames = torch.empty(b, n, 3, 3, device=dev, dtype=torch.float32)
        rc = L.pcl_frames_fwd(*_lib.pts_args(p), _lib.ptr(ln), b, n, K, int(bool(disambiguate_directions)), idx.data_ptr(),
                              curv.data_ptr(), frames.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_frames_fwd")
    return dict(curvatures=curv, frames=frames, idx=idx, points=p, lengths=ln)


class _FramesFunction(Function):
    @staticmethod
    def forward(ctx, points, lengths, K, disambiguate):
        ctx.in_meta = (points.dtype, points.device)
        ctx.set_materialize_grads(False)  # an unused output gives no work and no gradient through it
        r = frames_forward_raw(points, K, disambiguate, lengths)
        ctx.save_for_backward(r["points"], r["idx"], r["curvatures"], r["frames"])
        ctx.len = r["lengths"]
        return r["curvatures"], r["frames"]

    @staticmethod
    def backward(ctx, grad_curv, grad_frames):
        p, idx, curv, frames = ctx.saved_tensors
        b, n, _ = p.shape
        K = idx.shape[2]
        dev = p.device
        gc = None if grad_curv is None else grad_curv.to(device=dev, dtype=torch.float32).contiguous()
        gf = None if grad_frames is None else grad_frames.to(device=dev, dtype=torch.float32).contiguous()
        L = _lib.lib()
        with _lib.on_device(dev):
            gp = torch.empty(b, n, 3, device=dev, dtype=torch.float32)
            rc = L.pcl_frames_bwd(*_lib.pts_args(p), _lib.ptr(ctx.len), b, n, K, idx.data_ptr(), curv.data_ptr(),
                                  frames.data_ptr(), _lib.ptr(gc), _lib.ptr(gf), gp.data_ptr(), _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_frames_bwd")
        dt, d0 = ctx.in_meta
        return gp.to(device=d0, dtype=dt), None, None, None


def estimate_pointcloud_local_coord_frames(pointclouds, neighborhood_size=50, disambiguate_directions=True, *,
                                           use_symeig_workaround=True, lengths=None):
    """pytorch3d.ops.estimate_pointcloud_local_coord_frames [3P-memory] for a (N, P, 3) tensor of fp32 / fp16 / bf16 points
    (strided views are read in place) and optional int64 `lengths` (N,).  Returns (curvatures (N,P,3), frames (N,P,3,3)),
    both fp32: eigenvalues ascending and the matching eigenvectors as columns.  `use_symeig_workaround` is ignored.

    Raises ValueError like pytorch3d when the last dimension is not 3 or a cloud has at most `neighborhood_size` points,
    and when neighborhood_size is outside 1..knn_max_k().  Host synchronisation: with `lengths`, that size check reads
    them on the host, as pytorch3d does; without `lengths` nothing here synchronises."""
    return _FramesFunction.apply(pointclouds, lengths, neighborhood_size, bool(disambiguate_directions))


def estimate_pointcloud_normals(pointclouds, neighborhood_size=50, disambiguate_directions=True, *,
                                use_symeig_workaround=True, lengths=None):
    """pytorch3d.ops.estimate_pointcloud_normals [3P-memory]: column 0 of estimate_pointcloud_local_coord_frames, (N, P, 3)
    fp32 -- the direction of least variance of every point's neighbourhood."""
    _, frames = estimate_pointcloud_local_coord_frames(pointclouds, neighborhood_size, disambiguate_directions,
                                                       use_symeig_workaround=use_symeig_workaround, lengths=lengths)
    return frames[..., 0]
