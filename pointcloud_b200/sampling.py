"""Farthest point sampling and ball query -- B200 kernels behind the names the reference uses on the producer side
of the loss path (SURVEY.md 8f): `farthest_point_sample` / `query_ball_point` (models/pointnet2_utils.py:89-113) and
`sample_farthest_points` (pytorch3d call surface used at utils.py:90 and models/pointmlp.py:158)."""
import numbers

import torch

from . import _lib


def farthest_point_sample(xyz, npoint, start_idx=None, skip_origin=True):
    """xyz (B, N, 3+) -> sampled point indices (B, npoint), int64 like the reference wrapper (pointnet2_utils.py:89-90).
    N may be up to pcl_fps_max_points() (262144 points per cloud).

    `skip_origin=True` (default) is the behaviour of the kernel that wrapper calls (pointnet2_ops `furthest_point_sample`
    never selects a point with x^2+y^2+z^2 <= 1e-3 after the first [3P-memory]); `skip_origin=False` is the plain torch
    algorithm kept as a comment in pointnet2_utils.py:64-86 and pytorch3d's `sample_farthest_points`."""
    _lib.require_cuda()
    L = _lib.lib()
    xyz = _lib.as_points(xyz)
    b, n, c = xyz.shape
    assert c >= 3
    dev = xyz.device
    st = None if start_idx is None else start_idx.to(device=dev, dtype=torch.int32).contiguous()
    with _lib.on_device(dev):
        idx = torch.empty(b, int(npoint), device=dev, dtype=torch.int32)
        rc = L.pcl_fps(*_lib.pts_args(xyz), b, n, int(npoint), _lib.ptr(st), 1 if skip_origin else 0, idx.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_fps")
    return idx.long()


def _int_tensor(v, name, b, dev):
    """lengths / K argument -> int64 (b,) tensor on `dev`, or None."""
    if v is None:
        return None
    t = torch.as_tensor(v)
    if t.shape != (b,):
        raise ValueError(f"Expected {name} to be of shape (N,), got {tuple(t.shape)} for N={b}.")
    if t.dtype.is_floating_point or t.dtype == torch.bool:
        raise ValueError(f"{name} must hold integers")
    return t.to(device=dev, dtype=torch.int64).contiguous()


def fps_forward_raw(xyz, lengths=None, K=None, npoint=None, start_idx=None, skip_origin=False, cluster=0):
    """One pcl_fps_ragged call (include/pcl.h).  xyz (B, N, 3+); lengths and K: None or (B,) integer tensors; npoint:
    the output width (default: K, or max(K) for a tensor K).  `cluster` 0 = automatic, 1/2/4/8/16 forces a cluster size.
    Returns the int32 (B, npoint) indices: the FPS sequence over the first lengths[b] points, then -1 from slot
    min(lengths[b], K[b]) on."""
    _lib.require_cuda()
    L = _lib.lib()
    xyz = _lib.as_points(xyz)
    b, n, c = xyz.shape
    if c < 3:
        raise ValueError(f"expected at least 3 channels (xyz), got {c}")
    dev = xyz.device
    if npoint is None:
        if K is None:
            raise ValueError("npoint or K is needed")
        kk = K if isinstance(K, int) else torch.as_tensor(K)
        npoint = kk if isinstance(kk, int) else (int(kk.max()) if kk.numel() else 0)
    if isinstance(K, int):
        K = None if K >= npoint else torch.full((b,), K, dtype=torch.int64)
    ln, kt = _int_tensor(lengths, "lengths", b, dev), _int_tensor(K, "K", b, dev)
    st = None if start_idx is None else start_idx.to(device=dev, dtype=torch.int32).contiguous()
    with _lib.on_device(dev):
        idx = torch.empty(b, int(npoint), device=dev, dtype=torch.int32)
        rc = L.pcl_fps_ragged(*_lib.pts_args(xyz), _lib.ptr(ln), b, n, _lib.ptr(kt), int(npoint), _lib.ptr(st),
                              1 if skip_origin else 0, int(cluster), idx.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_fps_ragged")
    return idx


def sample_farthest_points(points, lengths=None, K=50, random_start_point=False):
    """pytorch3d.ops.sample_farthest_points(points, lengths, K, random_start_point) -> (sampled points (B, maxK, D),
    indices (B, maxK) int64).  The call surface and padding are pytorch3d's as recalled [3P-memory; pytorch3d is absent]:

    - `lengths` (B,): cloud b is points[b, :lengths[b]]; K is an int, a list / tuple or a (B,) tensor of per-cloud counts,
      the output width is max(K) (a CUDA K tensor costs one host read for it, as in pytorch3d);
    - slots from min(lengths[b], K[b]) on hold index -1 and zero points;
    - `random_start_point` starts cloud b at an index drawn uniformly from [0, lengths[b]).

    Distances use xyz only (the first three channels); pytorch3d uses ALL D channels -- the reference only passes xyz+rgb
    rows through it in the dataset transform (utils.py:90).  Without lengths and with an int K this keeps the
    behaviour of `farthest_point_sample`, including K > P, where index 0 repeats (pytorch3d would pad -1 there)."""
    if points.dim() != 3:
        raise ValueError(f"Expected points to be of shape (N, P, D), got {tuple(points.shape)}")
    b, p, d = points.shape
    ln = _int_tensor(lengths, "lengths", b, None)
    if isinstance(K, bool):
        raise ValueError("K must be an int, a list / tuple or a tensor")
    if isinstance(K, numbers.Integral) or (isinstance(K, torch.Tensor) and K.dim() == 0 and not K.dtype.is_floating_point
                                           and K.dtype != torch.bool):
        K = int(K)  # a scalar: Python / numpy integer or 0-dim integer tensor
        if K < 0:
            raise ValueError(f"K={K} must be >= 0")
        if lengths is None:
            start = None
            if random_start_point:
                start = torch.randint(0, points.shape[1], (points.shape[0],))
            idx = farthest_point_sample(points[:, :, :3], K, start_idx=start, skip_origin=False)
            gathered = torch.gather(points.to(idx.device), 1, idx.unsqueeze(-1).expand(-1, -1, points.shape[2]))
            return gathered, idx
        k_t = None
        width = K
    else:
        k_t = _int_tensor(K, "K", b, None)
        width, lo = 0, 0
        if b:
            lo, width = (int(v) for v in torch.stack(torch.aminmax(k_t)).cpu())  # one host read for a CUDA tensor
        if lo < 0:
            raise ValueError("K must be >= 0")
    _lib.require_cuda()
    pts = _lib.as_points(points)
    dev = pts.device
    ln = None if ln is None else ln.to(dev)
    start = None
    if random_start_point:
        n = ln.clamp(0, p) if ln is not None else torch.full((b,), p, device=dev, dtype=torch.int64)
        start = (torch.rand(b, device=dev, dtype=torch.float64) * n).long().clamp(max=(n - 1).clamp(min=0))
    idx = fps_forward_raw(pts[:, :, :3], ln, k_t, width, start_idx=start, skip_origin=False).long()
    keep = (idx >= 0).unsqueeze(-1)
    gathered = torch.gather(points.to(dev), 1, idx.clamp(min=0).unsqueeze(-1).expand(-1, -1, d))
    return torch.where(keep, gathered, torch.zeros((), dtype=gathered.dtype, device=dev)), idx


def query_ball_point(radius, nsample, xyz, new_xyz):
    """pointnet2_utils.py:93-113: (B, S, nsample) int64 indices of the first nsample points within `radius` of every
    centroid, padded with the first hit."""
    _lib.require_cuda()
    L = _lib.lib()
    xyz, new_xyz = _lib.as_points(xyz), _lib.as_points(new_xyz)
    b, n, _ = xyz.shape
    s = new_xyz.shape[1]
    dev = xyz.device
    r2 = float(torch.tensor(radius ** 2, dtype=torch.float32))  # the comparison happens in fp32 (sqrdists > radius ** 2)
    with _lib.on_device(dev):
        out = torch.empty(b, s, int(nsample), device=dev, dtype=torch.int32)
        rc = L.pcl_ball_query(*_lib.pts_args(xyz), *_lib.pts_args(new_xyz), b, n, s, r2, int(nsample), out.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_ball_query")
    return out.long()
