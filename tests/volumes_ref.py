"""float64 torch restatement of pytorch3d 0.7.2's add_points_features_to_volume_densities_features, restated from memory
[3P-memory].  Parity with pytorch3d itself is unpinned: THIS FILE IS THE SPECIFICATION the library is tested against
(include/pcl.h, "points to volumes", says the same in C terms).

  per axis (x -> W, y -> H, z -> D) with cloud size S (grid_sizes[b], or the padded size):
    t = ((p + 1) * (S - s) - o) * 0.5 in float32, every operation rounded;  (s, o) = (1, 0) with align_corners, else (0, 1)
  trilinear: f = floor(t), r = t - f; corner f + d (d in {0,1}^3) has weight w = m * ((wz * wy) * wx), w_a = d_a ? r_a : 1 - r_a
  nearest:   the voxel round_half_away_from_zero(t), weight m
  a vote lands at [b, :, z, y, x] when 0 <= index < min(S_axis, padded axis) on every axis; a point with m == 0
  is skipped entirely (m = mask[b, i], 1 without a mask), and one with a non-finite t has no corner in bounds.
  densities = initial + sum w;  features[c] = initial[c] + sum w * feature[c]  (a non-finite feature whose vote has w == 0
  adds nothing)
  rescale_features: features / densities.clamp(min_weight) (trilinear) or densities.clamp(1.0) (nearest)

Everything after t runs in float64; t enters as its float32 value with the derivative (S - s) / 2 (dr/dt = 1), so autograd
through this file gives the specified gradients: zero for the points in nearest mode and for non-finite points."""
import torch

F64 = torch.float64


def lattice(points, sizes, align_corners):
    """t (B,P,3) float32 in x, y, z order; sizes (B,3) int64 in (D, H, W) order."""
    s, o = (1, 0) if align_corners else (0, 1)
    S = sizes.flip(1)[:, None, :]                                    # (B,1,3) as (W, H, D)
    return ((points.detach().float() + 1) * (S - s).float() - o) * 0.5


def votes(points, mask, sizes, padded, mode, align_corners):
    """Every (point, corner) vote in point-major, corner-ascending order (corner k: dx = k & 1, dy = k >> 1 & 1, dz = k >> 2).
    -> (b, i, x, y, z, w, valid): int64 indices (0 where invalid), float64 weights (differentiable in the points), and
    whether the corner is in bounds.  An in-bounds corner of weight 0 adds exactly 0 but still carries dw/dt."""
    B, P, _ = points.shape
    dev = points.device
    sizes = sizes.to(dev)
    m = torch.ones(B, P, dtype=F64, device=dev) if mask is None else mask.to(dev).to(F64)
    t32 = lattice(points, sizes, align_corners)
    s = 1 if align_corners else 0
    k = (sizes.flip(1) - s).to(torch.float32).to(F64)[:, None, :] / 2  # d t / d p
    finite = torch.isfinite(t32).all(-1) & (m != 0)
    p64 = points.to(F64)
    t = t32.to(F64) + (p64 - p64.detach()) * k
    t = torch.where(finite[..., None], t, torch.zeros_like(t))       # non-finite points: no corner, no NaN gradient
    lim = torch.minimum(sizes.flip(1), torch.tensor(padded[::-1], device=dev))[:, None, :]  # (B,1,3) as (W, H, D)
    if mode == "trilinear":
        f = torch.floor(t.detach())
        r = t - f
        d = torch.tensor([[k & 1, (k >> 1) & 1, k >> 2] for k in range(8)], device=dev, dtype=F64)  # (8,3)
        idx = f[:, :, None, :] + d                                  # (B,P,8,3)
        wa = torch.where(d.bool(), r[:, :, None, :], 1 - r[:, :, None, :])
        w = m[:, :, None] * ((wa[..., 2] * wa[..., 1]) * wa[..., 0])  # (B,P,8)
    elif mode == "nearest":
        td = t.detach()
        idx = (torch.sign(td) * torch.floor(td.abs() + 0.5))[:, :, None, :]
        w = m[:, :, None] + 0 * t.sum(-1, keepdim=True)             # the points get a zero gradient
    else:
        raise ValueError(mode)
    valid = ((idx >= 0) & (idx < lim[:, :, None, :])).all(-1) & finite[:, :, None]
    idx = torch.where(valid[..., None], idx, torch.zeros_like(idx)).long()
    nc = idx.shape[2]
    bb = torch.arange(B, device=dev)[:, None, None].expand(B, P, nc)
    ii = torch.arange(P, device=dev)[None, :, None].expand(B, P, nc)
    return bb, ii, idx[..., 0], idx[..., 1], idx[..., 2], w, valid


def splat_ref(points_3d, points_features, volume_densities, volume_features=None, mode="trilinear", mask=None,
              grid_sizes=None, align_corners=True, stats=False):
    """The unscaled forward in float64: -> (features (B,C,D,H,W), densities (B,1,D,H,W)), differentiable in the points, the
    features and the initial volumes.  stats=True adds (n, abs_features, abs_densities): the number of votes per voxel and
    |initial| + sum |vote|, the scale of the accuracy bound (votes of weight 0 add exactly 0 and are not counted)."""
    B, P, C = points_features.shape
    D, H, W = volume_densities.shape[2:]
    dev = points_3d.device
    sizes = (torch.tensor([D, H, W], device=dev).expand(B, 3) if grid_sizes is None else grid_sizes.to(dev).long())
    bb, ii, x, y, z, w, valid = votes(points_3d, mask, sizes, (D, H, W), mode, align_corners)
    bb, ii, x, y, z, w = (a[valid] for a in (bb, ii, x, y, z, w))
    vox = ((bb * D + z) * H + y) * W + x
    f = points_features.to(dev).to(F64)[bb, ii]                      # (V, C)
    f = torch.where((w.detach() == 0)[:, None] & ~torch.isfinite(f), torch.zeros_like(f), f)
    dens0 = volume_densities.to(dev).to(F64).reshape(B * D * H * W)
    feat0 = (torch.zeros(B, C, D, H, W, dtype=F64, device=dev) if volume_features is None
             else volume_features.to(dev).to(F64))
    feat0 = feat0.permute(0, 2, 3, 4, 1).reshape(B * D * H * W, C)
    dens = dens0.index_add(0, vox, w)
    feat = feat0.index_add(0, vox, w[:, None] * f)
    out_f = feat.view(B, D, H, W, C).permute(0, 4, 1, 2, 3)
    out_d = dens.view(B, 1, D, H, W)
    if not stats:
        return out_f, out_d
    with torch.no_grad():
        n = torch.zeros(B * D * H * W, dtype=F64, device=dev).index_add(0, vox, (w != 0).to(F64)).view(B, 1, D, H, W)
        ad = dens0.abs().index_add(0, vox, w.abs()).view(B, 1, D, H, W)
        af = feat0.abs().index_add(0, vox, (w[:, None] * f).abs()).view(B, D, H, W, C).permute(0, 4, 1, 2, 3)
    return out_f, out_d, n, af, ad


def add_points_features_ref(points_3d, points_features, volume_densities, volume_features=None, mode="trilinear",
                            min_weight=1e-4, mask=None, grid_sizes=None, rescale_features=True, align_corners=True):
    """The public function's semantics in float64: -> (features, densities)."""
    feat, dens = splat_ref(points_3d, points_features, volume_densities, volume_features, mode, mask, grid_sizes,
                           align_corners)
    if rescale_features:
        feat = feat / dens.clamp(min_weight if mode == "trilinear" else 1.0)
    return feat, dens
