"""Points to volumes -- B200 drop-in for `pytorch3d.ops.add_points_features_to_volume_densities_features`.

The call surface and semantics are pytorch3d 0.7.2's as recalled ([3P-memory]; parity with pytorch3d itself is unpinned):
tests/volumes_ref.py restates them in float64 torch and is the specification; include/pcl.h ("points to volumes") says the
same in C terms.  Every point of cloud b votes into the voxel grid of its (D_b, H_b, W_b) = grid_sizes[b] (x -> W, y -> H,
z -> D) at the lattice coordinate t = ((p + 1) * (S - s) - o) * 0.5 (fp32, every operation rounded; (s, o) = (1, 0) with
align_corners, (0, 1) without): trilinear mode splats weight m * prod (d ? r : 1 - r) onto the 8 corners of floor(t),
nearest mode gives weight m to the voxel round(t), rounded half away from zero.  m is mask[b, i] used as a weight (a point
with m == 0 is skipped entirely, a non-finite coordinate contributes nothing).  A vote lands at [b, :, z, y, x] of the padded
tensor when 0 <= index < min(grid size, padded size) on every axis; voxels outside a cloud's grid keep their initial
values.  densities = initial + sum w; features[c] = initial[c] + sum w * feature[c]; with rescale_features the features are
divided by densities.clamp(min_weight) (trilinear) or densities.clamp(1.0) (nearest); the densities are returned unscaled.

Differences from pytorch3d, deliberate:
  - the outputs are new fp32 tensors and the initial volumes are never written;
  - grid_sizes on the device is never read back to the host;
  - there is no `_python=` switch, and no `add_pointclouds_to_volumes` (this library has no Pointclouds / Volumes types; a
    `mask` built from the cloud lengths plays that role, see INTEGRATION.md).

Gradients: points_features gets m * sum_corners w * grad_features[c]; points_3d, in trilinear mode only, gets
m * (S - s)/2 * sum_corners dw/dt * (grad_densities + sum_c feature[c] * grad_features[c]) with dr/dt = 1 (zeros in nearest
mode, where pytorch3d calls it undefined); the initial volumes get the upstream gradients unchanged; mask and grid_sizes get
none.  They come back in each input's dtype and on its device.
"""
import torch
from torch.autograd import Function

from . import _lib

_MODES = {"trilinear": 0, "nearest": 1}


def _check(points_3d, points_features, volume_densities, volume_features, mode, mask, grid_sizes):
    """pytorch3d's checks and messages, plus the shapes the kernels rely on.  Reads nothing from the device."""
    if points_3d.dim() != 3 or points_3d.shape[-1] != 3:
        raise ValueError(f"points_3d has to be of shape (minibatch, n_points, 3), got {tuple(points_3d.shape)}")
    if points_features.dim() != 3 or points_features.shape[2] < 1:
        raise ValueError(f"points_features has to be of shape (minibatch, n_points, C >= 1), got {tuple(points_features.shape)}")
    if volume_densities.dim() != 5:
        raise ValueError(f"volume_densities has to be of shape (minibatch, 1, D, H, W), got {tuple(volume_densities.shape)}")
    if volume_densities.shape[1] != 1:
        raise ValueError("Only one-dimensional densities are allowed.")
    if mode not in _MODES:
        raise ValueError('No such interpolation mode "%s"' % mode)
    b, p, c = points_features.shape
    if points_3d.shape[0] != b or volume_densities.shape[0] != b:
        raise ValueError(f"Batch sizes differ: points_3d {points_3d.shape[0]}, points_features {b}, "
                         f"volume_densities {volume_densities.shape[0]}")
    if points_3d.shape[1] != p:
        raise ValueError(f"points_3d has {points_3d.shape[1]} points per cloud, points_features {p}")
    if volume_features is not None:
        if volume_features.dim() != 5 or volume_features.shape[0] != b:
            raise ValueError(f"volume_features has to be of shape (minibatch, C, D, H, W), got {tuple(volume_features.shape)}")
        if volume_features.shape[1] != c:
            raise ValueError(f"volume_features has {volume_features.shape[1]} channels, points_features {c}")
        if volume_features.shape[2:] != volume_densities.shape[2:]:
            raise ValueError(f"volume_features grid {tuple(volume_features.shape[2:])} differs from volume_densities "
                             f"grid {tuple(volume_densities.shape[2:])}")
    if mask is not None and tuple(mask.shape) != (b, p):
        raise ValueError(f"mask has to be of shape (minibatch, n_points), got {tuple(mask.shape)}")
    if grid_sizes is not None and tuple(grid_sizes.shape) != (b, 3):
        raise ValueError(f"grid_sizes has to be of shape (minibatch, 3), got {tuple(grid_sizes.shape)}")


def _kernel_inputs(points_3d, points_features, mask, grid_sizes):
    """The kernels' views: points / features as strided CUDA fp32 / fp16 / bf16 (no copy when they already are), the mask
    as contiguous fp32, grid_sizes as contiguous int64, all on the points' device."""
    p = _lib.as_points(points_3d)
    dev = p.device
    f = _lib.as_points(points_features.to(dev))
    m = None if mask is None else mask.to(device=dev, dtype=torch.float32).contiguous()
    g = None if grid_sizes is None else grid_sizes.to(device=dev, dtype=torch.int64).contiguous()
    return p, f, m, g


def _fp32_clone(t, dev):
    out = torch.empty(t.shape, device=dev, dtype=torch.float32)
    out.copy_(t)
    return out


def points_to_volumes_forward_raw(points_3d, points_features, volume_densities, volume_features=None, mode="trilinear",
                                  mask=None, grid_sizes=None, align_corners=True):
    """pcl_points_to_volumes_fwd: the unscaled forward, without autograd.  Returns dict(features (B,C,D,H,W) fp32,
    densities (B,1,D,H,W) fp32): the initial volumes (cloned; zeros for volume_features=None) plus the votes."""
    _check(points_3d, points_features, volume_densities, volume_features, mode, mask, grid_sizes)
    p, f, m, g = _kernel_inputs(points_3d, points_features, mask, grid_sizes)
    dev = p.device
    b, n, c = f.shape
    d, h, w = volume_densities.shape[2:]
    with _lib.on_device(dev):
        dens = _fp32_clone(volume_densities, dev)
        if volume_features is None:
            feat = torch.zeros(b, c, d, h, w, device=dev, dtype=torch.float32)
        else:
            feat = _fp32_clone(volume_features, dev)
        rc = _lib.lib().pcl_points_to_volumes_fwd(*_lib.pts_args(p), *_lib.pts_args(f), _lib.ptr(m), _lib.ptr(g), b, n, c,
                                                  d, h, w, _MODES[mode], int(bool(align_corners)), dens.data_ptr(),
                                                  feat.data_ptr(), _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_points_to_volumes_fwd")
    return dict(features=feat, densities=dens)


class _PointsToVolumesFunction(Function):
    @staticmethod
    def forward(ctx, points_3d, points_features, volume_densities, volume_features, mask, grid_sizes, mode, align_corners):
        ctx.set_materialize_grads(False)  # an unused output gives no work and no gradient through it
        r = points_to_volumes_forward_raw(points_3d, points_features, volume_densities, volume_features, mode, mask,
                                          grid_sizes, align_corners)
        ctx.save_for_backward(points_3d, points_features, mask, grid_sizes)
        ctx.mode, ctx.align_corners, ctx.grid = mode, align_corners, tuple(volume_densities.shape[2:])
        ctx.vol_meta = (volume_densities.dtype, volume_densities.device,
                        None if volume_features is None else (volume_features.dtype, volume_features.device))
        return r["features"], r["densities"]

    @staticmethod
    def backward(ctx, grad_features, grad_densities):
        points_3d, points_features, mask, grid_sizes = ctx.saved_tensors
        p, f, m, g = _kernel_inputs(points_3d, points_features, mask, grid_sizes)
        dev = p.device
        b, n, c = f.shape
        gf = None if grad_features is None else grad_features.to(device=dev, dtype=torch.float32).contiguous()
        gd = None if grad_densities is None else grad_densities.to(device=dev, dtype=torch.float32).contiguous()
        d, h, w = ctx.grid
        want_p, want_f = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gp = gpf = None
        if (gd is not None or gf is not None) and (want_p or want_f):
            with _lib.on_device(dev):
                gp = torch.empty(b, n, 3, device=dev, dtype=torch.float32) if want_p else None
                gpf = torch.empty(b, n, c, device=dev, dtype=torch.float32) if want_f else None
                rc = _lib.lib().pcl_points_to_volumes_bwd(
                    *_lib.pts_args(p), *_lib.pts_args(f), _lib.ptr(m), _lib.ptr(g), b, n, c, d, h, w, _MODES[ctx.mode],
                    int(bool(ctx.align_corners)), _lib.ptr(gd), _lib.ptr(gf), _lib.ptr(gp), _lib.ptr(gpf),
                    _lib.stream_ptr(dev))
                _lib.check(rc, "pcl_points_to_volumes_bwd")
            gp = None if gp is None else gp.to(device=points_3d.device, dtype=points_3d.dtype)
            gpf = None if gpf is None else gpf.to(device=points_features.device, dtype=points_features.dtype)
        dt, dd, fmeta = ctx.vol_meta
        g_dens = None if grad_densities is None or not ctx.needs_input_grad[2] else grad_densities.to(device=dd, dtype=dt)
        g_feat = None
        if grad_features is not None and fmeta is not None and ctx.needs_input_grad[3]:
            g_feat = grad_features.to(device=fmeta[1], dtype=fmeta[0])
        return gp, gpf, g_dens, g_feat, None, None, None, None


def add_points_features_to_volume_densities_features(points_3d, points_features, volume_densities, volume_features=None,
                                                     mode="trilinear", min_weight=1e-4, mask=None, grid_sizes=None,
                                                     rescale_features=True, align_corners=True):
    """pytorch3d.ops.add_points_features_to_volume_densities_features [3P-memory]: splat ragged point clouds into voxel grids.

    points_3d (B,P,3) local volume coordinates in [-1, 1] and points_features (B,P,C): fp32 / fp16 / bf16 are read in place
    (strided views included), other floating types go through `.float()`.  volume_densities (B,1,D,H,W) and volume_features
    (B,C,D,H,W) or None (zeros) are the initial volumes; they are not modified.  mode "trilinear" or "nearest".  mask (B,P)
    bool / int / float or None: a per-point weight.  grid_sizes (B,3) int64 (D_b, H_b, W_b), CPU or CUDA, or None (the
    padded D, H, W).  Returns (volume_features (B,C,D,H,W), volume_densities (B,1,D,H,W)), both new fp32 tensors; see the
    module docstring for the semantics and the gradients.

    Raises ValueError like pytorch3d: points_3d's last dimension is not 3, volume_densities has more than one channel, an
    unknown mode, differing batch sizes, a channel count of volume_features other than C.  Nothing on the path reads device
    data on the host."""
    _check(points_3d, points_features, volume_densities, volume_features, mode, mask, grid_sizes)
    features, densities = _PointsToVolumesFunction.apply(points_3d, points_features, volume_densities, volume_features, mask,
                                                         grid_sizes, mode, bool(align_corners))
    if rescale_features:
        features = features / densities.clamp(min_weight if mode == "trilinear" else 1.0)
    return features, densities
